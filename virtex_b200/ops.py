"""Python-side launchers of the C-ABI kernels: torch tensors in, raw pointers out.

Every function launches on torch's current CUDA stream, never allocates and never synchronises.  There is no
fallback: a missing library or a non-CUDA tensor raises.
"""
import ctypes
from ctypes import c_float, c_int, c_int32, c_int64, c_uint32, c_void_p

import torch

from . import lib as L

P, I, I64, F, U32 = c_void_p, c_int, c_int64, c_float, c_uint32

_PROTOS = {
    "vtx_gemm": [P, P],
    "vtx_stem_im2col": [P, P, I, I, I, I, P],
    "vtx_stem_s2d": [P, P, I, I, I, P],
    "vtx_stem_s2d_w_pack": [P, P, I, P],
    "vtx_stem_s2d_w_unpack_add": [P, P, I, P],
    "vtx_im2col3x3": [P, P, I, I, I, I, I, P],
    "vtx_col2im3x3": [P, P, I, I, I, I, I, P],
    "vtx_subsample": [P, P, I, I, I, I, I, P],
    "vtx_upsample_add": [P, P, I, I, I, I, I, P],
    "vtx_bn_finalize": [P, F, P, P, P, P, P, F, F, I, P, I, P],
    "vtx_bn_act": [P, P, P, P, P, P, I64, I, I, P],
    "vtx_bn_finalize_act": [P, F, P, P, P, P, P, F, F, I, P, P, P, P, P, P, I64, I, I, P],
    "vtx_bn_bwd_finalize_apply": [P, P, F, P, P, P, P, P, P, P, P, P, P, P, P, P, I64, I, I, P],
    "vtx_bn_relu_maxpool": [P, P, P, P, I, I, I, I, P],
    "vtx_maxpool_bwd": [P, P, P, I, I, I, I, P],
    "vtx_bn_bwd_reduce": [P, P, P, P, P, P, P, P, I64, I, I, P],
    "vtx_bn_bwd_finalize": [P, P, F, P, P, P, I, P],
    "vtx_bn_bwd_apply": [P, P, P, P, P, P, P, P, P, P, P, I64, I, I, P],
    "vtx_conv_w_pack": [P, P, I, I, I, I, I, P],
    "vtx_conv_w_pack_dgrad": [P, P, I, I, P],
    "vtx_conv_w_unpack_add": [P, P, I, I, I, I, I, P],
    "vtx_conv_w_unpack_add_t": [P, P, I, I, I, I, P],
    "vtx_conv_w_jobs": [P, I, I, P],
    "vtx_cast_bf16": [P, P, I64, P],
    "vtx_nhwc_to_nchw_f32": [P, P, I, I, I, P],
    "vtx_embed_fwd": [P, P, P, P, P, P, P, P, P, I, I, I, I, F, F, P, U32, P],
    "vtx_embed_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, I, I, F, P, U32, P],
    "vtx_add_ln_fwd": [P, P, P, P, P, P, P, P, I, I, F, F, P, U32, I, P],
    "vtx_ln_bwd": [P, P, P, P, P, P, P, P, P, P, I, I, F, P, U32, I, P],
    "vtx_attn_fwd": [P, I64, P, I64, P, I64, P, I64, P, I, I, I, I, P, I, F, P, U32, P],
    "vtx_attn_bwd": [P, I64, P, I64, P, I64, P, I64, P, P, I64, P, I64, P, I64, I, I, I, I, P, I, F, P, U32, P],
    "vtx_gelu_dropout_fwd": [P, P, I64, F, P, U32, P],
    "vtx_gelu_dropout_bwd": [P, P, P, I64, F, P, U32, P],
    "vtx_count_valid": [P, I, I, I, I, P, P],
    "vtx_cross_entropy": [P, I64, P, I, I, I, I, I, P, P, I, P],
    "vtx_colsum": [P, I64, I, I, P, P],
    "vtx_argmax_rows": [P, I64, I, I, P, P],
    "vtx_decode_attn": [P, I64, P, P, I64, I64, P, I, I, P, I64, I, I, I, I, P],
    "vtx_beam_step": [P, I64, I, I, I, I, I, I, P, P, P, P, P, P, P],
    "vtx_beam_reorder": [P, P, P, P, I, I, P, P, I, I, I, P],
    "vtx_avgpool_fwd": [P, P, I, I, I, P],
    "vtx_avgpool_bwd": [P, P, I, I, I, P],
    "vtx_khot_xent": [P, I64, P, I, P, I, I, I, P, P, I64, P],
    "vtx_topk_rows": [P, I64, I, I, I, P, P],
    "vtx_image_resample": [P, P, P, P, P, P, I, I, P],
    "vtx_image_gray_sum": [P, P, P, P, I, I, P],
    "vtx_image_jitter_normalize": [P, P, P, P, P, P, I, I, P],
    "vtx_collate_tokens": [P, P, P, P, P, I, I, I, I64, P],
    "vtx_sumsq": [P, I64, P, P],
    "vtx_clip_coef": [P, I, F, P, P],
    "vtx_sgd_step": [P, P, P, P, P, P, I, P, P, F, F, P],
}

_fn = {}


def _get(name):
    f = _fn.get(name)
    if f is None:
        f = getattr(L.load(), name)
        f.argtypes = _PROTOS[name]
        f.restype = c_int
        _fn[name] = f
    return f


def exported_symbols():
    """All C-ABI entry points this module binds (used by the CPU test that checks the library exports them)."""
    return sorted(_PROTOS) + ["vtx_last_error", "vtx_version", "vtx_num_sms", "vtx_weight_job_block_elems", "vtx_sizeof_gemm",
                              "vtx_gemm_set_dynamic_schedule"]


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return 0 if t is None else t.data_ptr()


launch_count = 0          # number of kernels of this library launched so far (every entry point launches exactly one)
_gemm_profile = None      # when a list: (start_event, stop_event, flops, M, N, K, conv_mode, a_mn, b_mn) per GEMM launch


def call(name, *args):
    global launch_count
    rc = _get(name)(*args)
    if rc != 0:
        L.check(rc, name)
    launch_count += 1


def start_gemm_profile():
    global _gemm_profile
    _gemm_profile = []


def stop_gemm_profile():
    """Returns [(milliseconds, flops, M, N, K, conv_mode, a_mn, b_mn, extra_bytes)] for every GEMM launched since start;
    extra_bytes = what the epilogue reads besides A and B (residual tile, ReLU bit mask)."""
    global _gemm_profile
    torch.cuda.synchronize()
    out = [(a.elapsed_time(b),) + tuple(rest) for (a, b, *rest) in _gemm_profile]
    _gemm_profile = None
    return out


def num_sms():
    return L.load().vtx_num_sms()


def set_dynamic_gemm_schedule(on: bool):
    """Tile schedule of the persistent GEMM (include/virtex_b200.h): dynamic when another stream's kernels (NCCL) share
    the SMs with it, static otherwise."""
    L.check(L.load().vtx_gemm_set_dynamic_schedule(int(bool(on))), "vtx_gemm_set_dynamic_schedule")


# --------------------------------------------------------------------------------------------------------------- GEMM
_gemm_struct = L.VtxGemm()


def gemm(A, B, D, M, N, K, *, lda=None, ldb=None, ldd=None, a_mn=0, b_mn=0, bias=None, act=0, residual=None,
         ldr=0, stats=None, atomic=False, split_k=1, tile_n=0, conv=None, conv_mode=0, out_f32=None, residual_mask=None,
         conv_stride=1, conv_taps=0, tap_grid=None, out_view=None, d_ptr=None, bnr=None):
    """D[M,N] = epilogue(A . B^T) through the tcgen05 kernel; see include/virtex_b200.h (VtxGemm).
    bnr = (y, bnp, sums, mask or None[, y_ptr]): BN-backward reduction of the output fused into the epilogue."""
    g = _gemm_struct
    g.A, g.B, g.D = A.data_ptr(), B.data_ptr(), (D.data_ptr() if d_ptr is None else d_ptr)
    g.bias, g.residual, g.stats = _p(bias), _p(residual), _p(stats)
    g.residual_mask = _p(residual_mask)
    g.lda = A.stride(0) if lda is None else lda
    g.ldb = B.stride(0) if ldb is None else ldb
    g.ldd = D.stride(0) if ldd is None else ldd
    g.ldr = (residual.stride(0) if residual is not None else 0) if not ldr else ldr
    g.M, g.N, g.K = M, N, K
    g.a_mn, g.b_mn = a_mn, b_mn
    g.out_f32 = int(D.dtype == torch.float32) if out_f32 is None else int(out_f32)
    g.atomic, g.act, g.split_k, g.tile_n = int(atomic), act, split_k, tile_n
    g.alpha = 1.0
    if conv is not None:
        g.conv_n, g.conv_h, g.conv_w, g.conv_c = conv
    else:
        g.conv_n = g.conv_h = g.conv_w = g.conv_c = 0
    g.conv_mode = conv_mode
    g.conv_stride, g.conv_taps = conv_stride, conv_taps
    g.conv_taps_h, g.conv_taps_w, g.conv_pad = tap_grid if tap_grid is not None else (0, 0, 0)
    # out_view = (out_h, out_w, ldd_w, ldd_h, ldd_n): D (at d_ptr) is a strided sub-grid of a larger NHWC tensor
    g.conv_out_h, g.conv_out_w, g.ldd_w, g.ldd_h, g.ldd_n = out_view if out_view is not None else (0, 0, 0, 0, 0)
    if bnr is not None:
        g.bnr_y = bnr[0].data_ptr() if len(bnr) < 5 else bnr[4]
        g.bnr_bnp, g.bnr_sums, g.bnr_mask = bnr[1].data_ptr(), bnr[2].data_ptr(), _p(bnr[3])
        g.bnr_ldy = bnr[0].stride(0)
    else:
        g.bnr_y = g.bnr_bnp = g.bnr_sums = g.bnr_mask = None
        g.bnr_ldy = 0
    if _gemm_profile is None:
        call("vtx_gemm", ctypes.addressof(g), _stream())
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call("vtx_gemm", ctypes.addressof(g), _stream())
        e1.record()
        extra = (2 * M * N if residual is not None else 0) + (M * N // 8 if residual_mask is not None else 0)
        if bnr is not None:
            extra += 2 * M * N + (M * N // 8 if bnr[3] is not None else 0)
        _gemm_profile.append((e0, e1, 2.0 * M * N * K, M, N, K, conv_mode, a_mn, b_mn, extra))


def split_k_for(m_tiles_x_n_tiles, k_blocks, sms=None):
    """Split-K factor for reduction-heavy (wgrad) GEMMs; thresholds from the round-2 sweep (scripts/tune_gemm.py)."""
    sms = sms or num_sms()
    t = m_tiles_x_n_tiles
    if t >= sms:
        # one to three rounds of long-K tiles (vocabulary wgrad: 316 tiles x 120 k-blocks): two splits balance the tail
        return 2 if (t < 3 * sms and k_blocks >= 64) else 1
    if sms // t == 1:
        # 75..147 tiles: a single under-filled round; four splits measured best at 96 tiles (3H x H wgrad: 98 -> 60 us),
        # none at 128 tiles (FFN wgrads)
        return 4 if (t <= 0.7 * sms and k_blocks >= 16) else 1
    # about one wave of tiles: every extra split multiplies the fp32 atomic traffic of the epilogue
    return max(1, min(max(1, k_blocks // 4), sms // t))
