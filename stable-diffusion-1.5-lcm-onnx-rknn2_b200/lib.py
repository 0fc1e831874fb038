"""ctypes binding of libdreamlab_b200.so (the C-ABI in include/dreamlab_b200.h).

Fails loudly: a missing library or a failing call raises RuntimeError — nothing falls back to
PyTorch ops or the CPU.
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdreamlab_b200.so")

EPI_BF16, EPI_GEGLU, EPI_F32, EPI_U8_IMAGE, EPI_BF16_RELU = 0, 1, 2, 3, 4
ATTN_TC, ATTN_SIMT, ATTN_SIMT_CAUSAL = 0, 1, 2

EXPORTS = [
    "dl_abi_version", "dl_last_error", "dl_device_sm_count", "dl_igemm", "dl_igemm_plan_bn", "dl_fill_identity",
    "dl_groupnorm_workspace_bytes", "dl_groupnorm", "dl_layernorm", "dl_attention", "dl_attention_wide",
    "dl_debug_attention_trace",
    "dl_timestep_sinusoid", "dl_small_linear", "dl_upsample2x", "dl_im2col_s2", "dl_pack_latent",
    "dl_nchw_to_nhwc_f32", "dl_nhwc_to_nchw_f32", "dl_lcm_step", "dl_latent_pool8", "dl_softmax_rows",
    "dl_cfg_combine", "dl_groupnorm_split_workspace_bytes", "dl_groupnorm_stats", "dl_groupnorm_apply",
    "dl_im2col_s2_halo", "dl_tile_blend", "dl_image_crop_u8", "dl_igemm_tiles_per_image",
    "dl_groupnorm_finalize", "dl_groupnorm_finalize_channels", "dl_embed_tokens", "dl_act_bf16",
    "dl_peer_allgather", "dl_igemm_f32", "dl_groupnorm_f32", "dl_layernorm_f32", "dl_attention_f32", "dl_pack_latent_f32",
    "dl_im2col_s2_f32", "dl_softmax_rows_f32", "dl_small_linear_f32",
    "dl_png_stored_size", "dl_png_stored_workspace_bytes", "dl_png_stored", "dl_conv_tapsum",
    "dl_im2col_s2_pad01", "dl_im2col_s2_pad01_f32", "dl_pack_image_im2col", "dl_pack_image_im2col_f32",
    "dl_vae_sample_latents", "dl_pack_image_im2col_masked", "dl_pack_image_im2col_masked_f32",
    "dl_inpaint_latent_mask", "dl_pack_latent_inpaint", "dl_pack_latent_inpaint_f32", "dl_lcm_step_inpaint",
    "dl_taesd_latent_in", "dl_taesd_latent_in_f32", "dl_lcm_step_ex", "dl_lcm_step_inpaint_ex", "dl_sampler_step",
]


class IgemmDesc(C.Structure):
    _fields_ = [
        ("a0", C.c_void_p), ("a0_pix_stride", C.c_longlong), ("c0", C.c_int),
        ("a1", C.c_void_p), ("a1_pix_stride", C.c_longlong), ("c1", C.c_int),
        ("nimg", C.c_int), ("h", C.c_int), ("w", C.c_int), ("taps", C.c_int), ("tap_phase", C.c_int),
        ("wgt", C.c_void_p), ("ldw", C.c_longlong), ("n", C.c_int),
        ("out", C.c_void_p), ("ldo", C.c_longlong), ("out_x_stride", C.c_longlong),
        ("out_y_stride", C.c_longlong), ("out_img_stride", C.c_longlong),
        ("bias", C.c_void_p), ("rowadd", C.c_void_p), ("ld_rowadd", C.c_int),
        ("residual", C.c_void_p), ("ldr", C.c_longlong), ("identity", C.c_void_p),
        ("mode", C.c_int), ("alpha", C.c_float), ("bn", C.c_int),
        ("gn_partial", C.c_void_p), ("gn_cpg", C.c_int), ("gn_slots", C.c_int), ("gn_slot0", C.c_int),
        ("gn_rows_per_img", C.c_int),
        ("peer_out", C.c_void_p * 7), ("n_peer_out", C.c_int),
        ("in_rows", C.c_int), ("in_row0", C.c_int),
        ("row_stats_out", C.c_void_p), ("row_stats_slots", C.c_int),
        ("ln_stats", C.c_void_p), ("ln_slots", C.c_int), ("ln_colsum", C.c_void_p), ("ln_c", C.c_int),
        ("ln_eps", C.c_float),
    ]


class LcmCoeffs(C.Structure):
    _fields_ = [("sqrt_alpha_t", C.c_float), ("sqrt_beta_t", C.c_float), ("c_skip", C.c_float),
                ("c_out", C.c_float), ("sqrt_alpha_prev", C.c_float), ("sqrt_beta_prev", C.c_float)]


class LcmCoeffsEx(C.Structure):
    _fields_ = [("k", LcmCoeffs), ("prediction_type", C.c_int), ("clip_sample", C.c_int),
                ("clip_sample_range", C.c_float)]


class SamplerCoeffs(C.Structure):
    _fields_ = [("a_x", C.c_float), ("a_e", C.c_float), ("c_x", C.c_float), ("c_e", C.c_float), ("c_0", C.c_float),
                ("c_1", C.c_float), ("c_n", C.c_float), ("clip_sample", C.c_int), ("clip_sample_range", C.c_float)]


PRED_EPSILON, PRED_V, PRED_SAMPLE = 0, 1, 2
_PRED = {"epsilon": PRED_EPSILON, "v_prediction": PRED_V, "sample": PRED_SAMPLE}


def _coeffs_ex(coeffs, prediction_type, clip_range) -> LcmCoeffsEx:
    if prediction_type not in _PRED:
        raise RuntimeError(f"lcm_step: prediction_type must be one of {sorted(_PRED)}, got {prediction_type!r}")
    return LcmCoeffsEx(LcmCoeffs(*[float(v) for v in coeffs]), _PRED[prediction_type], int(clip_range is not None),
                       0.0 if clip_range is None else float(clip_range))


_lib = None
_lock = threading.Lock()
launch_count = 0      # number of native kernel-launching calls made (bench: gpu_launches)


def load() -> C.CDLL:
    """Load the native library (no build here: `__graft_entry__.build()` / build.py does that)."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"dreamlab_b200: native library missing: {LIB_PATH} "
                    "(run `python -c 'import __graft_entry__ as g; g.build()'`). "
                    "There is no CPU/PyTorch fallback.")
            lib = C.CDLL(LIB_PATH)
            lib.dl_last_error.restype = C.c_char_p
            lib.dl_groupnorm_workspace_bytes.restype = C.c_size_t
            lib.dl_groupnorm_workspace_bytes.argtypes = [C.c_int, C.c_int]
            lib.dl_igemm.argtypes = [C.POINTER(IgemmDesc), C.c_void_p]
            lib.dl_igemm_plan_bn.argtypes = [C.POINTER(IgemmDesc)]
            lib.dl_fill_identity.argtypes = [C.c_void_p, C.c_void_p]
            lib.dl_groupnorm.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
            lib.dl_igemm_tiles_per_image.argtypes = [C.c_int, C.c_int]
            lib.dl_groupnorm_finalize.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong,
                                                  C.c_void_p, C.c_void_p]
            lib.dl_groupnorm_finalize_channels.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                                           C.c_int, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p]
            lib.dl_groupnorm_split_workspace_bytes.restype = C.c_size_t
            lib.dl_groupnorm_split_workspace_bytes.argtypes = [C.c_int, C.c_int]
            lib.dl_groupnorm_stats.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
            lib.dl_groupnorm_apply.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, C.c_float, C.c_void_p, C.c_void_p, C.c_int,
                                               C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p]
            lib.dl_im2col_s2_halo.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_layernorm.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]
            lib.dl_attention_wide.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p,
                                              C.c_longlong, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_int,
                                              C.c_int, C.c_float, C.c_void_p]
            lib.dl_attention.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong,
                                         C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_longlong,
                                         C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float,
                                         C.c_int, C.c_int, C.c_void_p]
            lib.dl_timestep_sinusoid.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_small_linear.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.c_void_p]
            lib.dl_upsample2x.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p]
            lib.dl_im2col_s2.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.c_void_p]
            lib.dl_pack_latent.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_float,
                                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
            lib.dl_softmax_rows.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_nchw_to_nhwc_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p]
            lib.dl_nhwc_to_nchw_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                C.c_void_p]
            lib.dl_lcm_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_longlong, C.POINTER(LcmCoeffs), C.c_void_p]
            lib.dl_peer_allgather.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.POINTER(C.c_void_p),
                                              C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_longlong, C.c_void_p,
                                              C.c_void_p]
            lib.dl_igemm_f32.argtypes = [C.POINTER(IgemmDesc), C.c_void_p]
            lib.dl_groupnorm_f32.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_float, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_layernorm_f32.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_float, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]
            lib.dl_attention_f32.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p,
                                             C.c_longlong, C.c_int, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                                             C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p]
            lib.dl_pack_latent_f32.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.c_float, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p]
            lib.dl_im2col_s2_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_softmax_rows_f32.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_small_linear_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_embed_tokens.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_void_p, C.c_void_p]
            lib.dl_act_bf16.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p]
            lib.dl_tile_blend.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_int, C.c_void_p]
            lib.dl_image_crop_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_longlong, C.c_longlong, C.c_void_p]
            lib.dl_cfg_combine.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_longlong,
                                           C.c_void_p]
            lib.dl_latent_pool8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_void_p, C.c_void_p]
            lib.dl_conv_tapsum.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_int, C.c_void_p]
            lib.dl_im2col_s2_pad01.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                               C.c_void_p]
            lib.dl_im2col_s2_pad01_f32.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                                   C.c_void_p]
            for f in (lib.dl_pack_image_im2col, lib.dl_pack_image_im2col_f32):
                f.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_void_p,
                              C.c_void_p]
            lib.dl_vae_sample_latents.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                  C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_void_p,
                                                  C.c_void_p]
            for f in (lib.dl_pack_image_im2col_masked, lib.dl_pack_image_im2col_masked_f32):
                f.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_longlong, C.c_longlong,
                              C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p]
            lib.dl_inpaint_latent_mask.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
            for f in (lib.dl_pack_latent_inpaint, lib.dl_pack_latent_inpaint_f32):
                f.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
            lib.dl_lcm_step_inpaint.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                                                C.POINTER(LcmCoeffs), C.c_float, C.c_float, C.c_int, C.c_void_p]
            lib.dl_lcm_step_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_longlong, C.POINTER(LcmCoeffsEx), C.c_void_p]
            lib.dl_lcm_step_inpaint_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong,
                                                   C.POINTER(LcmCoeffsEx), C.c_float, C.c_float, C.c_int, C.c_void_p]
            lib.dl_sampler_step.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_longlong, C.POINTER(SamplerCoeffs),
                                            C.c_void_p]
            for f in (lib.dl_taesd_latent_in, lib.dl_taesd_latent_in_f32):
                f.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
            lib.dl_png_stored_size.restype = C.c_longlong
            lib.dl_png_stored_size.argtypes = [C.c_int, C.c_int]
            lib.dl_png_stored_workspace_bytes.restype = C.c_longlong
            lib.dl_png_stored_workspace_bytes.argtypes = [C.c_int, C.c_int]
            lib.dl_png_stored.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong,
                                          C.c_void_p, C.c_void_p]
            _lib = lib
    return _lib


_SYNC_DEBUG = os.environ.get("DREAMLAB_SYNC", "") not in ("", "0")


def _check(rc: int, what: str):
    if rc != 0:
        msg = load().dl_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"dreamlab_b200.{what} failed (status {rc}): {msg}")
    if _SYNC_DEBUG:                      # debugging aid: surface device faults at the faulting op
        try:
            torch.cuda.synchronize()
        except Exception as e:
            raise RuntimeError(f"dreamlab_b200.{what}: device fault after launch: {e}")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t):
    return None if t is None else t.data_ptr()


_identity = {}


def identity_matrix(device) -> "torch.Tensor":
    """Per-device 256x256 bf16 identity: B operand of the tensor-core residual add."""
    dev = torch.device(device)
    key = dev.index if dev.index is not None else torch.cuda.current_device()
    t = _identity.get(key)
    if t is None:
        with torch.cuda.device(key):
            t = torch.empty(256, 256, device=f"cuda:{key}", dtype=torch.bfloat16)
            _check(load().dl_fill_identity(t.data_ptr(), _stream()), "fill_identity")
            torch.cuda.current_stream().synchronize()
        _identity[key] = t
    return t


def _count(n=1):
    global launch_count
    launch_count += n


# ---- optional per-launch timing (bench.py roofline): CUDA events on the launching stream ----
_prof = None
_prof_detail = False


def profile_begin(detail: bool = False):
    """detail=True keys the result by kernel AND shape tag (per-shape efficiency tables)."""
    global _prof, _prof_detail
    _prof = []
    _prof_detail = detail


def profile_end():
    """-> {kernel: {"ms": total, "flops": total, "bytes": total, "n": launches}}"""
    global _prof
    torch.cuda.synchronize()
    out = {}
    for name, flops, nbytes, a, b, tag in _prof:
        if _prof_detail:
            name = f"{name} {tag}"
        d = out.setdefault(name, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
        d["ms"] += a.elapsed_time(b)
        d["flops"] += flops
        d["bytes"] += nbytes
        d["n"] += 1
    _prof = None
    return out


class _timed:
    __slots__ = ("name", "flops", "nbytes", "a", "tag")

    def __init__(self, name, flops=0.0, nbytes=0.0, tag=""):
        self.name, self.flops, self.nbytes, self.tag = name, flops, nbytes, tag

    def __enter__(self):
        if _prof is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if _prof is not None and exc[0] is None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _prof.append((self.name, self.flops, self.nbytes, self.a, b, self.tag))
        return False


def wait_for_driver(timeout_s: float = 20.0) -> None:
    """On a box without persistence mode the driver tears the GPU down when its last client exits; a process that
    starts inside that window gets a failing cuInit ("CUDA driver initialization failed"), and torch caches the
    resulting device count of 0 for the life of the process.  So before torch first touches CUDA: when a GPU device
    node exists, retry cuInit through the driver API until it succeeds (or the timeout passes; the caller's own
    check then fails loudly).  No GPU node (the CPU-only build container): returns at once."""
    import glob
    import time
    if not glob.glob("/dev/nvidia[0-9]*"):
        return
    try:
        cu = C.CDLL("libcuda.so.1")
    except OSError:
        return
    t0 = time.monotonic()
    while True:
        rc = cu.cuInit(0)
        if rc == 0 or rc == 100 or time.monotonic() - t0 > timeout_s:     # 100: CUDA_ERROR_NO_DEVICE
            return
        time.sleep(0.5)


def require_cuda():
    wait_for_driver()
    if not torch.cuda.is_available():
        raise RuntimeError("dreamlab_b200 needs a CUDA device (sm_100a); there is no CPU fallback")


# ------------------------------------------------------------------------------------------------
# thin wrappers: torch tensors in, launches on torch's current stream
# ------------------------------------------------------------------------------------------------
def igemm(a0, wgt, out, *, nimg, h, w, taps, n, c0=None, a0_stride=None, a1=None, c1=0,
          a1_stride=None, bias=None, rowadd=None, residual=None, ldr=None, ldo=None,
          mode=EPI_BF16, alpha=1.0, bn=0, tap_phase=-1, out_strides=None, in_rows=0, in_row0=0,
          gn_partial=None, gn_cpg=0, gn_slot0=0, gn_rows_per_img=0, peer_outs=None, row_stats=False, ln=None):
    """out[pixel, :n] = epilogue(conv/linear(a0 ‖ a1, wgt)).  a0/a1: NHWC bf16 (or [M, C] rows with
    nimg=1,h=1,w=M); wgt: bf16 [n, taps*(c0+c1)].
    row_stats=True: returns fp32 [rows, slots, 2] per-row (sum, sumsq) partials of the bf16 output (the
    LayerNorm statistics of the next GEMM).  ln=(stats, colsum, eps): LayerNorm of the A rows folded into this
    GEMM (wgt pre-multiplied by gamma, bias = the folded bias)."""
    d = IgemmDesc()
    c0 = a0.shape[-1] if c0 is None else c0
    d.a0, d.c0 = a0.data_ptr(), c0
    d.a0_pix_stride = a0.stride(-2) if a0_stride is None else a0_stride
    if a1 is not None:
        c1 = a1.shape[-1] if not c1 else c1
        d.a1, d.c1 = a1.data_ptr(), c1
        d.a1_pix_stride = a1.stride(-2) if a1_stride is None else a1_stride
    d.nimg, d.h, d.w, d.taps, d.tap_phase = nimg, h, w, taps, tap_phase
    if out_strides is not None:
        d.out_x_stride, d.out_y_stride, d.out_img_stride = out_strides
    d.wgt, d.n = wgt.data_ptr(), n
    d.ldw = wgt.stride(0) if wgt.dim() == 2 and wgt.stride(0) != wgt.shape[1] else 0
    d.out = out.data_ptr()
    d.ldo = out.stride(-2) if ldo is None else ldo
    d.bias = _ptr(bias)
    d.rowadd = _ptr(rowadd)
    d.ld_rowadd = rowadd.stride(0) if rowadd is not None else 0
    f32 = a0.dtype == torch.float32          # fp32 precision mode: CUDA-core kernels, same descriptor
    d.residual = _ptr(residual)
    d.ldr = (residual.stride(-2) if ldr is None else ldr) if residual is not None else 0
    d.identity = identity_matrix(residual.device).data_ptr() if (residual is not None and not f32) else None
    d.mode, d.alpha, d.bn = mode, alpha, bn
    d.in_rows, d.in_row0 = in_rows, in_row0
    if peer_outs:                      # device pointers (ints) of the same view in the peers' buffers
        for i, ptr in enumerate(peer_outs):
            d.peer_out[i] = ptr
        d.n_peer_out = len(peer_outs)
    if gn_partial is not None:         # [nimg, slots, groups, 2] fp32
        d.gn_partial, d.gn_cpg, d.gn_slots = gn_partial.data_ptr(), gn_cpg, gn_partial.shape[1]
        d.gn_slot0, d.gn_rows_per_img = gn_slot0, gn_rows_per_img
    m_rows = nimg * h * w
    stats_out = None
    if row_stats:
        bn_plan = load().dl_igemm_plan_bn(C.byref(d))
        slots = 2 * ((n + bn_plan - 1) // bn_plan)
        stats_out = torch.empty(m_rows, slots, 2, device=out.device, dtype=torch.float32)
        d.row_stats_out, d.row_stats_slots = stats_out.data_ptr(), slots
    if ln is not None:
        st, colsum, eps = ln
        d.ln_stats, d.ln_slots, d.ln_colsum = st.data_ptr(), st.shape[1], colsum.data_ptr()
        d.ln_c, d.ln_eps = c0, eps
    ncols = n // 2 if mode == EPI_GEGLU else n
    # algorithmic bytes: every operand once (activations, weights, residual) + the output
    nbytes = (2.0 * m_rows * (d.c0 + d.c1) + 2.0 * n * taps * (d.c0 + d.c1) + out.element_size() * m_rows * ncols
              + (2.0 * m_rows * n if residual is not None else 0.0))
    with _timed("igemm", 2.0 * nimg * h * w * n * taps * (d.c0 + d.c1), nbytes,
                tag=f"M={nimg * h * w} ({nimg}x{h}x{w}) N={n} K={taps}x{d.c0 + d.c1} mode={mode}"
                    f"{' +res' if residual is not None else ''}"):
        if f32:
            _check(load().dl_igemm_f32(C.byref(d), _stream()), "igemm_f32")
        else:
            _check(load().dl_igemm(C.byref(d), _stream()), "igemm")
    _count()
    return stats_out


def groupnorm_workspace_bytes(nimg, groups=32):
    return load().dl_groupnorm_workspace_bytes(nimg, groups)


def groupnorm(x0, out, gamma, beta, workspace, *, nimg, hw, groups=32, eps=1e-5, silu=True, x1=None):
    c0 = x0.shape[-1]
    c1 = x1.shape[-1] if x1 is not None else 0
    if x0.dtype == torch.float32:
        _check(load().dl_groupnorm_f32(x0.data_ptr(), c0, _ptr(x1), c1, nimg, hw, groups, eps, gamma.data_ptr(),
                                       beta.data_ptr(), int(silu), out.data_ptr(), _stream()), "groupnorm_f32")
        _count()
        return
    with _timed("groupnorm", 0.0, 4.0 * nimg * hw * (c0 + c1), tag=f"n={nimg} hw={hw} C={c0}+{c1}"):
        _check(load().dl_groupnorm(x0.data_ptr(), c0, _ptr(x1), c1, nimg, hw, groups, eps,
                                   gamma.data_ptr(), beta.data_ptr(), int(silu), out.data_ptr(),
                                   workspace.data_ptr(), _stream()), "groupnorm")
    _count(2)


def igemm_tiles_per_image(h, w):
    return load().dl_igemm_tiles_per_image(h, w)


def groupnorm_finalize(partial, stats, count):
    """partial fp32 [nimg, slots, groups, 2] (sum, sumsq) -> stats fp32 [nimg, groups, 2] (mean, M2)."""
    nimg, slots, groups, _ = partial.shape
    _check(load().dl_groupnorm_finalize(partial.data_ptr(), nimg, slots, groups, int(count), stats.data_ptr(),
                                        _stream()), "groupnorm_finalize")
    _count()


def groupnorm_finalize_channels(part0, part1, stats, groups, count):
    """part_k fp32 [nimg, slots_k, C_k, 2] per-channel (sum, sumsq) of the producer(s) of [x0 | x1] ->
    stats fp32 [nimg, groups, 2] (mean, M2)."""
    nimg, s0, c0, _ = part0.shape
    s1, c1 = (part1.shape[1], part1.shape[2]) if part1 is not None else (0, 0)
    _check(load().dl_groupnorm_finalize_channels(part0.data_ptr(), s0, c0, _ptr(part1), s1, c1, nimg, groups,
                                                 int(count), stats.data_ptr(), _stream()), "groupnorm_finalize_channels")
    _count()


def groupnorm_split_workspace_bytes(nimg, groups=32):
    return load().dl_groupnorm_split_workspace_bytes(nimg, groups)


def groupnorm_stats(x0, stats, workspace, *, nimg, hw, groups=32, x1=None):
    """stats fp32 [nimg, groups, 2] <- (mean, M2) of this rank's strip."""
    c0 = x0.shape[-1]
    c1 = x1.shape[-1] if x1 is not None else 0
    with _timed("groupnorm_stats", 0.0, 2.0 * nimg * hw * (c0 + c1), tag=f"n={nimg} hw={hw} C={c0}+{c1}"):
        _check(load().dl_groupnorm_stats(x0.data_ptr(), c0, _ptr(x1), c1, nimg, hw, groups,
                                         stats.data_ptr(), workspace.data_ptr(), _stream()),
               "groupnorm_stats")
    _count()


def groupnorm_apply(x0, out, gamma, beta, stats_all, *, nimg, hw, groups=32, eps=1e-5, silu=True,
                    x1=None, out_img_stride=0):
    """stats_all fp32 [nranks, nimg, groups, 2]; out may be the interior of a halo-padded buffer."""
    c0 = x0.shape[-1]
    c1 = x1.shape[-1] if x1 is not None else 0
    with _timed("groupnorm_apply", 0.0, 4.0 * nimg * hw * (c0 + c1), tag=f"n={nimg} hw={hw} C={c0}+{c1}"):
        _check(load().dl_groupnorm_apply(x0.data_ptr(), c0, _ptr(x1), c1, nimg, hw, groups, eps,
                                         gamma.data_ptr(), beta.data_ptr(), int(silu),
                                         stats_all.data_ptr(), stats_all.shape[0], out.data_ptr(),
                                         out_img_stride, _stream()), "groupnorm_apply")
    _count()


def layernorm(x, out, gamma, beta, eps=1e-5):
    rows = x.numel() // x.shape[-1]
    if x.dtype == torch.float32:
        _check(load().dl_layernorm_f32(x.data_ptr(), rows, x.shape[-1], eps, gamma.data_ptr(), beta.data_ptr(),
                                       out.data_ptr(), _stream()), "layernorm_f32")
        _count()
        return
    with _timed("layernorm", 0.0, 4.0 * x.numel()):
        _check(load().dl_layernorm(x.data_ptr(), rows, x.shape[-1], eps, gamma.data_ptr(),
                                   beta.data_ptr(), out.data_ptr(), _stream()), "layernorm")
    _count()


def attention(q, k, v, out, *, batch, sq, skv, heads, d, dh_stride, ldq, ldk, ldv, ldo, scale,
              impl=ATTN_TC, v_ones=False):
    if q.dtype == torch.float32:
        _check(load().dl_attention_f32(q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, dh_stride,
                                       out.data_ptr(), ldo, batch, sq, skv, heads, d, scale,
                                       int(impl == ATTN_SIMT_CAUSAL), _stream()), "attention_f32")
        _count()
        return
    with _timed("attention", 4.0 * batch * heads * sq * skv * d,
                tag=f"B={batch} Sq={sq} Skv={skv} h={heads} d={d}"):
        _check(load().dl_attention(q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, dh_stride,
                                   out.data_ptr(), ldo, batch, sq, skv, heads, d, scale, impl,
                                   int(v_ones), _stream()), "attention")
    _count()


def attention_wide(q, k, v, out, *, batch, sq, skv, d, ldq, ldk, ldv, ldo, scale):
    """One-head flash attention for head dims up to 512 (the VAE mid block); bf16 only."""
    with _timed("attention_wide", 4.0 * batch * sq * skv * d,
                tag=f"B={batch} Sq={sq} Skv={skv} d={d}"):
        _check(load().dl_attention_wide(q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, out.data_ptr(), ldo,
                                        batch, sq, skv, d, scale, _stream()), "attention_wide")
    _count()


def timestep_sinusoid(t, out):
    _check(load().dl_timestep_sinusoid(t.data_ptr(), t.numel(), out.shape[-1], out.data_ptr(),
                                       _stream()), "timestep_sinusoid")
    _count()


def small_linear(x, w, out, bias=None, add=None, silu_in=False, silu_out=False):
    m, k = x.shape
    n = w.shape[0]
    if w.dtype == torch.float32:
        _check(load().dl_small_linear_f32(x.data_ptr(), m, k, w.data_ptr(), _ptr(bias), _ptr(add), n,
                                          int(silu_in), int(silu_out), out.data_ptr(), _stream()),
               "small_linear_f32")
        _count()
        return
    _check(load().dl_small_linear(x.data_ptr(), m, k, w.data_ptr(), _ptr(bias), _ptr(add), n,
                                  int(silu_in), int(silu_out), out.data_ptr(), _stream()),
           "small_linear")
    _count((m + 15) // 16)


def upsample2x(x, out, *, nimg, h, w):
    with _timed("upsample2x", 0.0, 10.0 * x.numel()):
        _check(load().dl_upsample2x(x.data_ptr(), nimg, h, w, x.shape[-1], out.data_ptr(), _stream()),
               "upsample2x")
    _count()


def im2col_s2(x, cols, *, nimg, h, w):
    if x.dtype == torch.float32:
        _check(load().dl_im2col_s2_f32(x.data_ptr(), nimg, h, w, x.shape[-1], cols.data_ptr(), _stream()),
               "im2col_s2_f32")
        _count()
        return
    with _timed("im2col_s2", 0.0, 2.0 * x.numel() + 2.0 * cols.numel()):
        _check(load().dl_im2col_s2(x.data_ptr(), nimg, h, w, x.shape[-1], cols.data_ptr(), _stream()),
               "im2col_s2")
    _count()


def im2col_s2_halo(x, cols, *, nimg, in_rows, in_row0, h, w):
    with _timed("im2col_s2", 0.0, 2.0 * x.numel() + 2.0 * cols.numel()):
        _check(load().dl_im2col_s2_halo(x.data_ptr(), nimg, in_rows, in_row0, h, w, x.shape[-1],
                                        cols.data_ptr(), _stream()), "im2col_s2_halo")
    _count()


def im2col_s2_pad01(x, cols, *, nimg, h, w):
    """Downsample2D(padding=0) of the VAE encoder: bottom / right zero pad, then conv3x3 stride 2."""
    if x.dtype == torch.float32:
        _check(load().dl_im2col_s2_pad01_f32(x.data_ptr(), nimg, h, w, x.shape[-1], cols.data_ptr(), _stream()),
               "im2col_s2_pad01_f32")
        _count()
        return
    with _timed("im2col_s2_pad01", 0.0, 2.0 * x.numel() + 2.0 * cols.numel()):
        _check(load().dl_im2col_s2_pad01(x.data_ptr(), nimg, h, w, x.shape[-1], cols.data_ptr(), _stream()),
               "im2col_s2_pad01")
    _count()


def pack_image_im2col(img, out, mask=None):
    """img: u8 [n,h,w,3] (a view with unit channel and 3-byte pixel stride: a tile window of a canvas is fine);
    out: bf16 or fp32 [n*h*w, 64] conv_in im2col operand (K = tap*3 + c, zero padded).
    mask (inpainting): u8 [n,h,w] with unit pixel stride (a window too); pixels with m >= 128 read as 0.0."""
    n, h, w, c = img.shape
    if c != 3 or img.dtype != torch.uint8 or img.stride(3) != 1 or img.stride(2) != 3:
        raise RuntimeError("pack_image_im2col: u8 [n,h,w,3] with packed RGB pixels expected")
    nbytes = float(img.numel()) + out.element_size() * out.numel()
    if mask is None:
        fn = load().dl_pack_image_im2col_f32 if out.dtype == torch.float32 else load().dl_pack_image_im2col
        with _timed("pack_image_im2col", 0.0, nbytes):
            _check(fn(img.data_ptr(), n, h, w, img.stride(1), img.stride(0), out.data_ptr(), _stream()),
                   "pack_image_im2col")
        _count()
        return
    if tuple(mask.shape) != (n, h, w) or mask.dtype != torch.uint8 or mask.stride(2) != 1:
        raise RuntimeError(f"pack_image_im2col: mask u8 [{n},{h},{w}] with unit pixel stride expected")
    fn = load().dl_pack_image_im2col_masked_f32 if out.dtype == torch.float32 else load().dl_pack_image_im2col_masked
    with _timed("pack_image_im2col_masked", 0.0, nbytes + mask.numel()):
        _check(fn(img.data_ptr(), mask.data_ptr(), n, h, w, img.stride(1), img.stride(0), mask.stride(1),
                  mask.stride(0), out.data_ptr(), _stream()), "pack_image_im2col_masked")
    _count()


def inpaint_latent_mask(mask, out):
    """mask u8 [n, 8h, 8w] (contiguous) -> out fp32 [n, h, w]: the binarised pixel (8i, 8j) of each latent."""
    n, h, w = out.shape
    if tuple(mask.shape) != (n, 8 * h, 8 * w) or mask.dtype != torch.uint8 or not mask.is_contiguous():
        raise RuntimeError(f"inpaint_latent_mask: contiguous u8 [{n},{8 * h},{8 * w}] expected")
    _check(load().dl_inpaint_latent_mask(mask.data_ptr(), n, h, w, out.data_ptr(), _stream()), "inpaint_latent_mask")
    _count()


def pack_latent_inpaint(latents, mask, masked, out, repeat=1):
    """latents / masked fp32 NHWC [n,h,w,4], mask fp32 [n,h,w] -> out bf16 or fp32 [repeat*n, h, w, 64]:
    [latents | mask | masked | 0...], the n images written `repeat` times."""
    npix = mask.numel()
    if latents.numel() != 4 * npix or masked.numel() != 4 * npix or out.numel() != 64 * npix * repeat:
        raise RuntimeError("pack_latent_inpaint: shapes do not match")
    fn = load().dl_pack_latent_inpaint_f32 if out.dtype == torch.float32 else load().dl_pack_latent_inpaint
    _check(fn(latents.data_ptr(), mask.data_ptr(), masked.data_ptr(), npix, repeat, out.data_ptr(), _stream()),
           "pack_latent_inpaint")
    _count()


def lcm_step_inpaint(eps, x, noise, image_latents, noise0, mask, x_next, denoised, coeffs, add_noise, last):
    """`lcm_step` + the 4-channel UNet's blend; add_noise = (sqrt_alpha, sqrt_one_minus_alpha) of the next timestep
    (ignored on the last step, where the blend target is image_latents itself)."""
    k = LcmCoeffs(*[float(v) for v in coeffs])
    _check(load().dl_lcm_step_inpaint(eps.data_ptr(), x.data_ptr(), _ptr(noise), image_latents.data_ptr(),
                                      _ptr(noise0), mask.data_ptr(), x_next.data_ptr(), denoised.data_ptr(),
                                      mask.numel(), C.byref(k), float(add_noise[0]), float(add_noise[1]), int(last),
                                      _stream()), "lcm_step_inpaint")
    _count()


def lcm_step_inpaint_ex(model_output, x, noise, image_latents, noise0, mask, x_next, denoised, coeffs, add_noise,
                        last, prediction_type="epsilon", clip_range=None):
    """`lcm_step_inpaint` with the x0 of `lcm_step_ex` (prediction_type, clamp of x0 to [-clip_range, clip_range])."""
    k = _coeffs_ex(coeffs, prediction_type, clip_range)
    _check(load().dl_lcm_step_inpaint_ex(model_output.data_ptr(), x.data_ptr(), _ptr(noise), image_latents.data_ptr(),
                                         _ptr(noise0), mask.data_ptr(), x_next.data_ptr(), denoised.data_ptr(),
                                         mask.numel(), C.byref(k), float(add_noise[0]), float(add_noise[1]),
                                         int(last), _stream()), "lcm_step_inpaint_ex")
    _count()


def vae_sample_latents(moments, eps_s, eps_n, out, *, scaling_factor, sqrt_alpha, sqrt_one_minus_alpha,
                       mean_out=None):
    """moments fp32 NHWC [n,h,w,8]; eps_s / eps_n fp32 NCHW [n,4,h,w]; out (mean_out) fp32 NHWC [n,h,w,4]."""
    n, h, w, _ = moments.shape
    _check(load().dl_vae_sample_latents(moments.data_ptr(), eps_s.data_ptr(), eps_n.data_ptr(), n, h, w,
                                        float(scaling_factor), float(sqrt_alpha), float(sqrt_one_minus_alpha),
                                        out.data_ptr(), _ptr(mean_out), _stream()), "vae_sample_latents")
    _count()


def pack_latent(x, out, *, cin, scale=1.0, mat=None, vec=None):
    npix = x.numel() // cin
    if out.dtype == torch.float32:
        _check(load().dl_pack_latent_f32(x.data_ptr(), npix, cin, out.shape[-1], scale, _ptr(mat), _ptr(vec),
                                         out.data_ptr(), _stream()), "pack_latent_f32")
        _count()
        return
    _check(load().dl_pack_latent(x.data_ptr(), npix, cin, out.shape[-1], scale, _ptr(mat),
                                 _ptr(vec), out.data_ptr(), _stream()), "pack_latent")
    _count()


def taesd_latent_in(latents, out):
    """latents fp32 NHWC [n,h,w,4] -> out bf16 or fp32 [n,h,w,64]: tanh(x / 3) * 3 in channels 0-3, zeros after
    (the input of the AutoencoderTiny decoder's first conv)."""
    npix = latents.numel() // 4
    if (latents.dtype != torch.float32 or latents.shape[-1] != 4 or not latents.is_contiguous()
            or out.shape[-1] != 64 or out.numel() != 64 * npix or not out.is_contiguous()):
        raise RuntimeError("taesd_latent_in: contiguous fp32 [..., 4] latents and a contiguous [..., 64] output expected")
    fn = load().dl_taesd_latent_in_f32 if out.dtype == torch.float32 else load().dl_taesd_latent_in
    with _timed("taesd_latent_in", 0.0, 16.0 * npix + out.element_size() * out.numel()):
        _check(fn(latents.data_ptr(), npix, out.data_ptr(), _stream()), "taesd_latent_in")
    _count()


def softmax_rows(scores, out):
    rows, cols = scores.shape
    if out.dtype == torch.float32:
        _check(load().dl_softmax_rows_f32(scores.data_ptr(), rows, cols, out.data_ptr(), _stream()),
               "softmax_rows_f32")
        _count()
        return
    with _timed("softmax_rows", 0.0, 6.0 * scores.numel()):
        _check(load().dl_softmax_rows(scores.data_ptr(), rows, cols, out.data_ptr(), _stream()),
               "softmax_rows")
    _count()


def nchw_to_nhwc_f32(x, out):
    n, c, h, w = x.shape
    _check(load().dl_nchw_to_nhwc_f32(x.data_ptr(), n, c, h * w, out.data_ptr(), _stream()),
           "nchw_to_nhwc_f32")
    _count()


def nhwc_to_nchw_f32(x, out):
    n, c, h, w = out.shape
    _check(load().dl_nhwc_to_nchw_f32(x.data_ptr(), n, c, h * w, out.data_ptr(), _stream()),
           "nhwc_to_nchw_f32")
    _count()


def lcm_step(eps, x, noise, x_next, denoised, coeffs):
    k = LcmCoeffs(*[float(v) for v in coeffs])
    _check(load().dl_lcm_step(eps.data_ptr(), x.data_ptr(), _ptr(noise), x_next.data_ptr(),
                              denoised.data_ptr(), x.numel(), C.byref(k), _stream()), "lcm_step")
    _count()


def lcm_step_ex(model_output, x, noise, x_next, denoised, coeffs, prediction_type="epsilon", clip_range=None):
    """`LCMScheduler.step` of the model's scheduler config: x0 from the model output by prediction_type ("epsilon",
    "v_prediction", "sample"), clamped to [-clip_range, clip_range] unless clip_range is None."""
    k = _coeffs_ex(coeffs, prediction_type, clip_range)
    _check(load().dl_lcm_step_ex(model_output.data_ptr(), x.data_ptr(), _ptr(noise), x_next.data_ptr(),
                                 denoised.data_ptr(), x.numel(), C.byref(k), _stream()), "lcm_step_ex")
    _count()


def peer_barrier(stage_ptrs, flag_ptrs, rank, slot_bytes, state):
    """dl_peer_allgather with an empty message: all ranks' earlier work (and its peer writes) is done."""
    R = len(stage_ptrs)
    sp = (C.c_void_p * R)(*stage_ptrs)
    fp = (C.c_void_p * R)(*flag_ptrs)
    _check(load().dl_peer_allgather(None, None, 0, sp, fp, R, rank, slot_bytes, state.data_ptr(), _stream()),
           "peer_barrier")
    _count()


def peer_allgather(src, dst, stage_ptrs, flag_ptrs, rank, slot_bytes, state):
    """src: contiguous local message; dst: [R, *src.shape]; stage_ptrs / flag_ptrs: per-rank device
    pointers (ints) of the symmetric staging buffers and signal pads."""
    R = len(stage_ptrs)
    sp = (C.c_void_p * R)(*stage_ptrs)
    fp = (C.c_void_p * R)(*flag_ptrs)
    _check(load().dl_peer_allgather(src.data_ptr(), dst.data_ptr(), src.numel() * src.element_size(), sp, fp, R,
                                    rank, slot_bytes, state.data_ptr(), _stream()), "peer_allgather")
    _count()


def embed_tokens(ids, tok_emb, pos_emb, out, seq):
    """ids int64 [n]; tok_emb bf16 [V, D]; pos_emb bf16 [seq, D]; out bf16 [n, D]."""
    _check(load().dl_embed_tokens(ids.data_ptr(), tok_emb.data_ptr(), pos_emb.data_ptr(), ids.numel(), seq,
                                  tok_emb.shape[0], tok_emb.shape[1], out.data_ptr(), _stream()), "embed_tokens")
    _count()


def act_bf16(x, out, mode):
    _check(load().dl_act_bf16(x.data_ptr(), out.data_ptr(), x.numel(), mode, _stream()), "act_bf16")
    _count()


def tile_blend(a, b, extent, vertical):
    """fp32 NHWC tiles; b's first `extent` rows (vertical) / columns blended in place with a's last."""
    n, ha, wa, c = a.shape
    _, hb, wb, _ = b.shape
    _check(load().dl_tile_blend(a.data_ptr(), b.data_ptr(), n, ha, wa, hb, wb, c, extent, int(vertical),
                                _stream()), "tile_blend")
    _count()


def image_crop_u8(src, crop_h, crop_w, dst_window):
    """src fp32 [n,hs,ws,c] -> u8 canvas window (a view [n, >=crop_h, >=crop_w, c] of the canvas)."""
    n, hs, ws, c = src.shape
    _check(load().dl_image_crop_u8(src.data_ptr(), n, hs, ws, c, crop_h, crop_w, dst_window.data_ptr(),
                                   dst_window.stride(1), dst_window.stride(0), _stream()), "image_crop_u8")
    _count()


def cfg_combine(eps_uncond, eps_text, guidance_scale, out):
    _check(load().dl_cfg_combine(eps_uncond.data_ptr(), eps_text.data_ptr(), float(guidance_scale),
                                 out.data_ptr(), out.numel(), _stream()), "cfg_combine")
    _count()


def sampler_step(out_uncond, out_text, guidance_scale, x, x0_prev, noise, x_next, x0, coeffs, clip_range=None):
    """One step of a guided-model sampler (`scheduler.py` schedules): e = out_uncond + guidance_scale * (out_text -
    out_uncond) (out_text None: e = out_uncond), x0 = a_x x + a_e e clamped to [-clip_range, clip_range] unless
    clip_range is None, x_next = c_x x + c_e e + c_0 x0 + c_1 x0_prev + c_n noise.  coeffs = (a_x, a_e, c_x, c_e,
    c_0, c_1, c_n); fp32 tensors of x's size."""
    n = x.numel()
    for name, t in (("out_uncond", out_uncond), ("out_text", out_text), ("x0_prev", x0_prev), ("noise", noise),
                    ("x_next", x_next), ("x0", x0)):
        if t is not None and (t.numel() != n or t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError(f"sampler_step: {name} must be a contiguous fp32 tensor of {n} elements")
    k = SamplerCoeffs(*[float(v) for v in coeffs], int(clip_range is not None),
                      0.0 if clip_range is None else float(clip_range))
    with _timed("sampler_step", 0.0, 4.0 * n * (4 + (out_text is not None) + (x0_prev is not None)
                                               + (noise is not None))):
        _check(load().dl_sampler_step(out_uncond.data_ptr(), _ptr(out_text), float(guidance_scale), x.data_ptr(),
                                      _ptr(x0_prev), _ptr(noise), x_next.data_ptr(), x0.data_ptr(), n, C.byref(k),
                                      _stream()), "sampler_step")
    _count()


def latent_pool8(lat_nhwc, out_f16):
    n, h, w, c = lat_nhwc.shape
    _check(load().dl_latent_pool8(lat_nhwc.data_ptr(), n, h, w, c, out_f16.data_ptr(), _stream()),
           "latent_pool8")
    _count()


def png_stored_size(h, w) -> int:
    return int(load().dl_png_stored_size(h, w))


def png_stored(img_u8, out=None):
    """img u8 NHWC [n,h,w,3] on the device -> (u8 [n, stride] with one PNG file per row, file size)."""
    n, h, w, c = img_u8.shape
    if c != 3 or img_u8.dtype != torch.uint8 or not img_u8.is_contiguous():
        raise RuntimeError("png_stored: contiguous u8 [n,h,w,3] expected")
    size = png_stored_size(h, w)
    stride = (size + 3) & ~3
    if out is None:
        out = torch.empty(n, stride, device=img_u8.device, dtype=torch.uint8)
    ws = torch.empty(load().dl_png_stored_workspace_bytes(n, h), device=img_u8.device, dtype=torch.uint8)
    _check(load().dl_png_stored(img_u8.data_ptr(), n, h, w, out.data_ptr(), out.stride(0), ws.data_ptr(), _stream()),
           "png_stored")
    _count(2)
    return out, size


def conv_tapsum(y, bias, out):
    """y fp32 [n,h,w,ldy] tap-major partial products, bias fp32 [nout], out u8 or fp32 [n,h,w,nout]."""
    n, h, w, ldy = y.shape
    nout = out.shape[-1]
    with _timed("conv_tapsum", 0.0, 4.0 * y.numel() + out.element_size() * out.numel()):
        _check(load().dl_conv_tapsum(y.data_ptr(), n, h, w, ldy, nout, bias.data_ptr(), out.data_ptr(),
                                     int(out.dtype == torch.uint8), _stream()), "conv_tapsum")
    _count()
