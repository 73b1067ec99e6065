"""ctypes binding of the C ABI in include/bcosk.h (libbcosk.so).

The header is the single source of truth: `bcosk_igemm_params` is parsed from it, and the result is
checked against `bcosk_sizeof_igemm_params()` of the loaded library.  There is NO fallback: if the
library is missing, cannot be loaded, or the device is not sm_100, the callers raise.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, List, Tuple

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
HEADER = os.path.join(ROOT, "include", "bcosk.h")
# $BCOSK_LIB: an alternative build of the same sources (experiment variants compiled with -D knobs); never a fallback
LIB_PATH = os.environ.get("BCOSK_LIB") or os.path.join(PKG, "libbcosk.so")

_CT = {
    "int32_t": C.c_int32, "uint32_t": C.c_uint32, "int64_t": C.c_int64, "uint16_t": C.c_uint16,
    "float": C.c_float, "int": C.c_int,
}


def _parse_struct(src: str, name: str, defines: Dict[str, int]) -> List[Tuple[str, object]]:
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), src, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields: List[Tuple[str, object]] = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(const\s+)?(\w+)\s*(\*?)\s*(.*)", decl)
        base, ptr, names = m.group(2), m.group(3), m.group(4)
        for nm in names.split(","):
            nm = nm.strip()
            is_ptr = bool(ptr) or nm.startswith("*")
            nm = nm.lstrip("* ")
            arr = re.match(r"(\w+)\[(\w+)\]", nm)
            if is_ptr:
                fields.append((nm, C.c_void_p))
            elif arr:
                n = defines.get(arr.group(2)) or int(arr.group(2))
                fields.append((arr.group(1), _CT[base] * n))
            else:
                fields.append((nm, _CT[base]))
    return fields


def _parse_header():
    with open(HEADER) as fh:
        src = fh.read()
    defines = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(BCOSK_\w+)\s+\(?(-?\d+)\)?", src)}
    protos = re.findall(r"^(?:int|const char\*)\s+(bcosk_\w+)\(", src, re.M)
    return defines, _parse_struct(src, "bcosk_igemm_params", defines), _parse_struct(src, "bcosk_wgrad_params", defines), protos


DEFINES, _FIELDS, _WGRAD_FIELDS, EXPORTS = _parse_header()
globals().update(DEFINES)  # BCOSK_OK, BCOSK_MODE_FWD, ...


class IgemmParams(C.Structure):
    _fields_ = _FIELDS

    def set_ptr(self, name: str, tensor) -> None:
        setattr(self, name, None if tensor is None else tensor.data_ptr())


class WgradParams(C.Structure):
    _fields_ = _WGRAD_FIELDS


class BcoskError(RuntimeError):
    pass


_lib = None


def load():
    """Load libbcosk.so (building is the job of `bcos_b200.build` / `__graft_entry__.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise BcoskError(f"{LIB_PATH} not found - run `python -m bcos_b200.build` (there is no CPU/PyTorch fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.bcosk_last_error.restype = C.c_char_p
    for name in EXPORTS:
        if not hasattr(lib, name):
            raise BcoskError(f"libbcosk.so does not export {name}")
    if lib.bcosk_sizeof_igemm_params() != C.sizeof(IgemmParams):
        raise BcoskError(f"bcosk_igemm_params layout mismatch: lib {lib.bcosk_sizeof_igemm_params()} vs "
                         f"binding {C.sizeof(IgemmParams)}")
    if lib.bcosk_sizeof_wgrad_params() != C.sizeof(WgradParams):
        raise BcoskError(f"bcosk_wgrad_params layout mismatch: lib {lib.bcosk_sizeof_wgrad_params()} vs binding {C.sizeof(WgradParams)}")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().bcosk_last_error().decode(errors="replace")
        raise BcoskError(f"{what} failed (rc={rc}): {msg}")


def require_device() -> None:
    """Raise unless the current CUDA device can run the sm_100a kernels."""
    import torch
    if not torch.cuda.is_available():
        raise BcoskError("bcos_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    if not load().bcosk_device_supported():
        raise BcoskError("bcos_b200 kernels are built for sm_100a (B200) only")


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


DTYPE_CODE = {"bf16": 1, "fp16": 0}


def torch_dtype(code: int):
    import torch
    return torch.bfloat16 if code == 1 else torch.float16


# ------------------------------------------------------------------------------------------------
# thin wrappers (device tensors in, nothing allocated here)
# ------------------------------------------------------------------------------------------------
def igemm(p: IgemmParams) -> None:
    check(load().bcosk_igemm(C.byref(p), _stream()), "bcosk_igemm")


def igemm_hp_config(p: IgemmParams) -> Tuple[int, ...]:
    """(CTAs per SM the kernel is built for, threads, dynamic shared memory bytes, CTAs per SM the occupancy API reports,
    registers per thread, local memory bytes per thread) of a parity-mode launch, without launching it (include/bcosk.h
    bcosk_igemm_hp_config)."""
    info = (C.c_int32 * 6)()
    check(load().bcosk_igemm_hp_config(C.byref(p), info), "bcosk_igemm_hp_config")
    return tuple(int(v) for v in info)


def debug_a_tile(p: IgemmParams, tile_m: int, chunk: int, out) -> None:
    check(load().bcosk_debug_a_tile(C.byref(p), tile_m, chunk, _p(out), _stream()), "bcosk_debug_a_tile")


def _f6(vals):
    return (C.c_float * 6)(*[float(v) for v in vals])


def _is_u8(x) -> bool:
    import torch
    nb, c, h, w = x.shape
    assert x.is_contiguous()
    if x.dtype == torch.uint8:
        assert c == 3, "uint8 input must be RGB [nb, 3, h, w]"
        return True
    assert x.dtype == torch.float32 and c == 6, "float input must be fp32 [nb, 6, h, w] = [x, 1-x]"
    return False


def _pixel_pitches(t):
    """(row pitch, image pitch) in pixels of an NHWC tensor or view (pixels themselves must be contiguous)."""
    assert t.stride(3) == 1 and t.stride(2) == t.shape[3], "pixels of an NHWC view must be contiguous"
    assert t.stride(1) % t.stride(2) == 0 and t.stride(0) % t.stride(2) == 0
    return t.stride(1) // t.stride(2), t.stride(0) // t.stride(2)


def input_prep_s2d(x, mean6, inv_std6, out, cp, planes, dtype, sq) -> None:
    nb, _, h, w = x.shape
    fn = load().bcosk_input_prep_s2d_u8 if _is_u8(x) else load().bcosk_input_prep_s2d
    rp, ip = _pixel_pitches(out)
    check(fn(_p(x), nb, h, w, _f6(mean6), _f6(inv_std6), _p(out), cp, planes, dtype, _p(sq), rp, ip, _stream()),
          "bcosk_input_prep_s2d")


def patch_inv_norm(sq, parts, nb, h, w, kh, kw, stride, pad, eps_in, eps_out, inv_norm, op, oq) -> None:
    check(load().bcosk_patch_inv_norm(_p(sq), parts, nb, h, w, kh, kw, stride, pad, C.c_float(eps_in), C.c_float(eps_out),
                                      _p(inv_norm), op, oq, _stream()), "bcosk_patch_inv_norm")


def pixel_sqsum(x, rows, c, planes, plane_stride, ld, dtype, sq) -> None:
    check(load().bcosk_pixel_sqsum(_p(x), C.c_int64(rows), c, planes, plane_stride, ld, dtype, _p(sq), _stream()),
          "bcosk_pixel_sqsum")


def avgpool_fwd(x, nb, h, w, c, planes, k, stride, pad, y, op, oq, dtype, sq) -> None:
    check(load().bcosk_avgpool_fwd(_p(x), nb, h, w, c, planes, k, stride, pad, _p(y), op, oq, dtype, _p(sq), _stream()),
          "bcosk_avgpool_fwd")


def avgpool_bwd_mul(gy, nb, h, w, c, planes, k, stride, pad, op, oq, gain, gain_f32, gx, dtype, gain_sqrt_scale=None) -> None:
    rp, ip = _pixel_pitches(gx)
    check(load().bcosk_avgpool_bwd_mul(_p(gy), nb, h, w, c, planes, k, stride, pad, op, oq, _p(gain), int(gain_f32), _p(gx),
                                       dtype, rp, ip, _p(gain_sqrt_scale), _stream()), "bcosk_avgpool_bwd_mul")


def explanation_rgba(grad6, x, smooth, percentile, tmp, out) -> None:
    nb, _, h, w = grad6.shape
    assert tmp.numel() >= 2 * nb * h * w + nb and tuple(out.shape) == (nb, h, w, 4)
    fn = load().bcosk_explanation_rgba_u8 if _is_u8(x) else load().bcosk_explanation_rgba
    check(fn(_p(grad6), _p(x), nb, h, w, int(smooth), C.c_float(percentile), _p(tmp), _p(out), _stream()),
          "bcosk_explanation_rgba")


def localisation_scores(attr, smooth, cell, negate, tmp, out) -> None:
    nt, c, h, w = attr.shape
    regions = (h // cell) * (w // cell)
    assert tmp.numel() >= 2 * nt * h * w + nt * regions and tuple(out.shape) == (nt, regions)
    check(load().bcosk_localisation_scores(_p(attr), nt, c, h, w, int(smooth), int(cell), int(bool(negate)), _p(tmp), _p(out),
                                           _stream()), "bcosk_localisation_scores")


def maxout_bcos_fwd(lin, inv_norm, rows, o, m, scale_mode, b_exp, y, gain, amax) -> None:
    check(load().bcosk_maxout_bcos_fwd(_p(lin), _p(inv_norm), C.c_int64(rows), o, m, scale_mode, C.c_float(b_exp), _p(y), _p(gain),
                                       _p(amax), _stream()), "bcosk_maxout_bcos_fwd")


def maxout_scatter(src, amax, rows, o, m, planes, dtype, dst) -> None:
    check(load().bcosk_maxout_scatter(_p(src), _p(amax), C.c_int64(rows), o, m, planes, dtype, _p(dst), _stream()),
          "bcosk_maxout_scatter")


def gap_logits(fc, nb, npix, ncls, inv_temp, bias, logits, pred) -> None:
    check(load().bcosk_gap_logits(_p(fc), nb, npix, ncls, C.c_float(inv_temp), C.c_float(bias), _p(logits), _p(pred),
                                  _stream()), "bcosk_gap_logits")


def fc_seed_dgrad(target, gain_fc, gain_f32, w_fc, nb, npix, ncls, c, inv_temp, seed_scale, mul1, mul1_f32, out1, mask2,
                  out2, planes, dtype) -> None:
    check(load().bcosk_fc_seed_dgrad(_p(target), _p(gain_fc), int(gain_f32), _p(w_fc), nb, npix, ncls, c,
                                     C.c_float(inv_temp), C.c_float(seed_scale), _p(mul1), int(mul1_f32), _p(out1),
                                     _p(mask2), _p(out2), planes, dtype, _stream()), "bcosk_fc_seed_dgrad")


def contrib_map_s2d(g, x, nb, h, w, cp, inv_std6, out_scale, cmap, grad6) -> None:
    fn = load().bcosk_contrib_map_s2d_u8 if _is_u8(x) else load().bcosk_contrib_map_s2d
    check(fn(_p(g), _p(x), nb, h, w, cp, _f6(inv_std6), C.c_float(out_scale), _p(cmap), _p(grad6), _stream()),
          "bcosk_contrib_map_s2d")


def channel_affine(x, rows, c, alpha, beta, relu, y, dtype) -> None:
    check(load().bcosk_channel_affine(_p(x), C.c_int64(rows), c, _p(alpha), _p(beta), int(relu), _p(y), dtype, _stream()),
          "bcosk_channel_affine")


def mul(a, b, n, out, dtype) -> None:
    check(load().bcosk_mul(_p(a), _p(b), C.c_int64(n), _p(out), dtype, _stream()), "bcosk_mul")


def nchw_to_nhwc16(x, out, cp, planes, dtype, mul=None, sq=None) -> None:
    nb, c, h, w = x.shape
    assert x.dtype.is_floating_point and x.element_size() == 4 and x.is_contiguous()
    check(load().bcosk_nchw_to_nhwc16(_p(x), nb, c, h, w, _p(out), cp, planes, dtype, _p(mul),
                                      0 if mul is None else mul.shape[-1], _p(sq), _stream()), "bcosk_nchw_to_nhwc16")


# ---- fused SimpleViT plan (csrc/bcosk_vit.cu)
def vit_patchify(x, p, mean6, inv_std6, out, planes, dtype, sq) -> None:
    nb, _, h, w = x.shape
    fn = load().bcosk_vit_patchify_u8 if _is_u8(x) else load().bcosk_vit_patchify
    check(fn(_p(x), nb, h, w, p, _f6(mean6), _f6(inv_std6), _p(out), planes, dtype, _p(sq), _stream()), "bcosk_vit_patchify")


def vit_contrib_map(g, x, p, inv_std6, out_scale, cmap, grad6) -> None:
    nb, _, h, w = x.shape
    fn = load().bcosk_vit_contrib_map_u8 if _is_u8(x) else load().bcosk_vit_contrib_map
    check(fn(_p(g), _p(x), nb, h, w, p, _f6(inv_std6), C.c_float(out_scale), _p(cmap), _p(grad6), _stream()), "bcosk_vit_contrib_map")


def vit_ln_fwd(x, rows, d, planes, w, eps, y, rstd, sq, dtype, out_planes=0) -> None:
    check(load().bcosk_vit_ln_fwd(_p(x), C.c_int64(rows), d, planes, out_planes, _p(w), C.c_float(eps), _p(y), _p(rstd), _p(sq), dtype, _stream()),
          "bcosk_vit_ln_fwd")


def vit_ln_bwd(g, G_in, rows, d, w, rstd, G_out, gain, ghat, dtype) -> None:
    import torch
    check(load().bcosk_vit_ln_bwd(_p(g), int(g.dtype == torch.float32), _p(G_in), C.c_int64(rows), d, _p(w), _p(rstd), _p(G_out), _p(gain),
                                  int(gain is not None and gain.dtype == torch.float32), _p(ghat), dtype, _stream()), "bcosk_vit_ln_bwd")


def vit_ln_bwd_full(g, x, planes, G_in, rows, d, w, rstd, G_out, gain, ghat, dtype) -> None:
    import torch
    check(load().bcosk_vit_ln_bwd_full(_p(g), int(g.dtype == torch.float32), _p(x), planes, _p(G_in), C.c_int64(rows), d, _p(w), _p(rstd), _p(G_out),
                                       _p(gain), int(gain is not None and gain.dtype == torch.float32), _p(ghat), dtype, _stream()),
          "bcosk_vit_ln_bwd_full")


def vit_quickgelu_fwd(u, rows, d, planes, a, sq, gain, dtype) -> None:
    import torch
    check(load().bcosk_vit_quickgelu_fwd(_p(u), C.c_int64(rows), d, planes, _p(a), _p(sq), _p(gain),
                                         int(gain is not None and gain.dtype == torch.float32), dtype, _stream()), "bcosk_vit_quickgelu_fwd")


def vit_attention_bwd_full(qkv, planes, g, batch, n, heads, dim_head, scale, out, dtype) -> None:
    check(load().bcosk_vit_attention_bwd_full(_p(qkv), planes, _p(g), batch, n, heads, dim_head, C.c_float(scale), _p(out), dtype, _stream()),
          "bcosk_vit_attention_bwd_full")


def vit_gelu_fwd(u, rows, d, planes, a, sq, gain, dtype) -> None:
    import torch
    check(load().bcosk_vit_gelu_fwd(_p(u), C.c_int64(rows), d, planes, _p(a), _p(sq), _p(gain),
                                    int(gain is not None and gain.dtype == torch.float32), dtype, _stream()), "bcosk_vit_gelu_fwd")


def vit_attention(qkv, planes, g, batch, n, heads, dim_head, scale, backward, out, dtype, tc=True) -> None:
    fn = load().bcosk_vit_attention_tc if tc else load().bcosk_vit_attention
    check(fn(_p(qkv), planes, _p(g), batch, n, heads, dim_head, C.c_float(scale), int(backward), _p(out), dtype,
                                     _stream()), "bcosk_vit_attention")


# ---- fused DenseNet plan (csrc/bcosk_dense.cu)
def dense_bn_relu_fwd(x, rows, c, planes, x_ld, x_plane_stride, alpha, relu, y, sq, maskbits, dtype) -> None:
    check(load().bcosk_dense_bn_relu_fwd(_p(x), C.c_int64(rows), c, planes, x_ld, x_plane_stride, _p(alpha), int(relu), _p(y), _p(sq),
                                         _p(maskbits), dtype, _stream()), "bcosk_dense_bn_relu_fwd")


def dense_bn_relu_bwd(g, rows, c, alpha, maskbits, G, g_ld, accumulate, dtype) -> None:
    import torch
    check(load().bcosk_dense_bn_relu_bwd(_p(g), int(g.dtype == torch.float32), C.c_int64(rows), c, _p(alpha), _p(maskbits), _p(G), g_ld,
                                         int(accumulate), dtype, _stream()), "bcosk_dense_bn_relu_bwd")


def dense_slice_cast(G, g_ld, col0, rows, c, gain, scale, out, dtype) -> None:
    import torch
    check(load().bcosk_dense_slice_cast(_p(G), g_ld, col0, C.c_int64(rows), c, _p(gain), int(gain is not None and gain.dtype == torch.float32),
                                        C.c_float(scale), _p(out), dtype, _stream()), "bcosk_dense_slice_cast")


def copy_rows_2d(dst_ptr, dst_pitch, src_ptr, src_pitch, width, rows) -> None:
    check(load().bcosk_copy_rows_2d(C.c_void_p(dst_ptr), C.c_int64(dst_pitch), C.c_void_p(src_ptr), C.c_int64(src_pitch), C.c_int64(width),
                                    C.c_int64(rows), _stream()), "bcosk_copy_rows_2d")


# ---- attention-pool head inside the fused CLIP plan (csrc/bcosk_head.cu)
def sgemm_batched(trans_a, trans_b, m, n, k, a_ptr, lda, stride_a, b_ptr, ldb, stride_b, c_ptr, ldc, stride_c, batch, alpha) -> None:
    check(load().bcosk_sgemm_batched(int(trans_a), int(trans_b), m, n, k, C.c_void_p(a_ptr), C.c_int64(lda), C.c_int64(stride_a),
                                     C.c_void_p(b_ptr), C.c_int64(ldb), C.c_int64(stride_b), C.c_void_p(c_ptr), C.c_int64(ldc),
                                     C.c_int64(stride_c), batch, C.c_float(alpha), _stream()), "bcosk_sgemm_batched")


def sgemm_batched_acc(trans_a, trans_b, m, n, k, a_ptr, lda, stride_a, b_ptr, ldb, stride_b, c_ptr, ldc, stride_c, batch, alpha) -> None:
    check(load().bcosk_sgemm_batched_acc(int(trans_a), int(trans_b), m, n, k, C.c_void_p(a_ptr), C.c_int64(lda), C.c_int64(stride_a),
                                         C.c_void_p(b_ptr), C.c_int64(ldb), C.c_int64(stride_b), C.c_void_p(c_ptr), C.c_int64(ldc),
                                         C.c_int64(stride_c), batch, C.c_float(alpha), _stream()), "bcosk_sgemm_batched_acc")


def softmax_bwd(p, dp, rows, n, ds) -> None:
    check(load().bcosk_softmax_bwd(_p(p), _p(dp), C.c_int64(rows), n, _p(ds), _stream()), "bcosk_softmax_bwd")


def head_tokens(x, nb, npix, c, planes, dtype, tokens) -> None:
    check(load().bcosk_head_tokens(_p(x), nb, npix, c, planes, dtype, _p(tokens), _stream()), "bcosk_head_tokens")


def row_softmax(s, rows, n) -> None:
    check(load().bcosk_row_softmax(_p(s), C.c_int64(rows), n, _stream()), "bcosk_row_softmax")


def seed_from_tokens(g_tokens, nb, npix, c, scale, mul1, out1, mask2, mul2, out2, planes, dtype) -> None:
    import torch
    check(load().bcosk_seed_from_tokens(_p(g_tokens), nb, npix, c, C.c_float(scale), _p(mul1),
                                        int(mul1 is not None and mul1.dtype == torch.float32), _p(out1), _p(mask2), _p(mul2),
                                        int(mul2 is not None and mul2.dtype == torch.float32), _p(out2), planes, dtype, _stream()),
          "bcosk_seed_from_tokens")


def stem_im2col_u8(x, k, stride, pad, mean6, inv_std6, a_scale, out, kp, inv_norm, dtype) -> None:
    nb, _, h, w = x.shape
    check(load().bcosk_stem_im2col_u8(_p(x), nb, h, w, k, stride, pad, _f6(mean6), _f6(inv_std6), C.c_float(a_scale), _p(out), kp, _p(inv_norm),
                                      dtype, _stream()), "bcosk_stem_im2col_u8")


def zero_insert_nhwc(src, dst, stride) -> None:
    nb, oh, ow, e = src.shape
    check(load().bcosk_zero_insert_nhwc(_p(src), nb, oh, ow, e, _p(dst), dst.shape[1], dst.shape[2], stride, _stream()), "bcosk_zero_insert_nhwc")


def nhwc_scatter_nchw_f32(y, nb, c, oh, ow, planes, dtype, out, stride) -> None:
    import torch
    check(load().bcosk_nhwc_scatter_nchw_f32(_p(y), int(y.dtype == torch.float32), nb, c, oh, ow, y.shape[-1], planes, dtype, _p(out),
                                             out.shape[2], out.shape[3], stride, _stream()), "bcosk_nhwc_scatter_nchw_f32")


def pixel_sqsum_nchw_f32(x, sq) -> None:
    nb, c, h, w = x.shape
    check(load().bcosk_pixel_sqsum_nchw_f32(_p(x), nb, c, C.c_int64(h * w), _p(sq), _stream()), "bcosk_pixel_sqsum_nchw_f32")


def seed_from_nchw(g, seed_scale, mul1, out1, mask2, mul2, out2, planes, dtype) -> None:
    import torch
    nb, c, h, w = g.shape
    assert g.dtype == torch.float32 and g.is_contiguous()
    check(load().bcosk_seed_from_nchw(_p(g), nb, c, h, w, C.c_float(seed_scale), _p(mul1),
                                      int(mul1 is not None and mul1.dtype == torch.float32), _p(out1), _p(mask2), _p(mul2),
                                      int(mul2 is not None and mul2.dtype == torch.float32), _p(out2), planes, dtype, _stream()),
          "bcosk_seed_from_nchw")


def nhwc_to_nchw_f32(y, nb, c, h, w, planes, dtype, out) -> None:
    import torch
    check(load().bcosk_nhwc_to_nchw_f32(_p(y), int(y.dtype == torch.float32), nb, c, h, w, y.shape[-1], planes, dtype, _p(out),
                                        _stream()), "bcosk_nhwc_to_nchw_f32")


def scale_bias_nchw(x, nb, c, hw, alpha, beta, smul, sadd, relu, out) -> None:
    check(load().bcosk_scale_bias_nchw(_p(x), nb, c, C.c_int64(hw), _p(alpha), _p(beta), C.c_float(smul), C.c_float(sadd),
                                       int(relu), _p(out), _stream()), "bcosk_scale_bias_nchw")


def channel_stats_nchw(x, nb, c, hw, mean, var) -> None:
    check(load().bcosk_channel_stats_nchw(_p(x), nb, c, C.c_int64(hw), _p(mean), _p(var), _stream()), "bcosk_channel_stats_nchw")


def layernorm_fwd(x, rows, d, w, b, eps, y, rstd) -> None:
    check(load().bcosk_layernorm_fwd(_p(x), C.c_int64(rows), d, _p(w), _p(b), C.c_float(eps), _p(y), _p(rstd), _stream()),
          "bcosk_layernorm_fwd")


def layernorm_explain_bwd(gy, rows, d, w, rstd, gx) -> None:
    check(load().bcosk_layernorm_explain_bwd(_p(gy), C.c_int64(rows), d, _p(w), _p(rstd), _p(gx), _stream()),
          "bcosk_layernorm_explain_bwd")


def groupnorm_fwd(x, nb, c, hw, groups, w, b, eps, centred, y, rstd) -> None:
    check(load().bcosk_groupnorm_fwd(_p(x), nb, c, C.c_int64(hw), groups, _p(w), _p(b), C.c_float(eps), int(centred), _p(y),
                                     _p(rstd), _stream()), "bcosk_groupnorm_fwd")


def groupnorm_explain_bwd(gy, nb, c, hw, groups, w, rstd, centred, gx) -> None:
    check(load().bcosk_groupnorm_explain_bwd(_p(gy), nb, c, C.c_int64(hw), groups, _p(w), _p(rstd), int(centred), _p(gx),
                                             _stream()), "bcosk_groupnorm_explain_bwd")


def positionnorm_fwd(x, nb, c, hw, w, b, eps, centred, y, rstd) -> None:
    check(load().bcosk_positionnorm_fwd(_p(x), nb, c, C.c_int64(hw), _p(w), _p(b), C.c_float(eps), int(centred), _p(y),
                                        _p(rstd), _stream()), "bcosk_positionnorm_fwd")


def positionnorm_explain_bwd(gy, nb, c, hw, w, rstd, centred, gx) -> None:
    check(load().bcosk_positionnorm_explain_bwd(_p(gy), nb, c, C.c_int64(hw), _p(w), _p(rstd), int(centred), _p(gx),
                                                _stream()), "bcosk_positionnorm_explain_bwd")


def l2norm_rows(x, rows, d, y, inv) -> None:
    check(load().bcosk_l2norm_rows(_p(x), C.c_int64(rows), d, _p(y), _p(inv), _stream()), "bcosk_l2norm_rows")


def row_scale(x, rows, d, s, y) -> None:
    check(load().bcosk_row_scale(_p(x), C.c_int64(rows), d, _p(s), _p(y), _stream()), "bcosk_row_scale")


def gelu_gate(x, g, n, y) -> None:
    check(load().bcosk_gelu_gate(_p(x), _p(g), C.c_int64(n), _p(y), _stream()), "bcosk_gelu_gate")


def attention(qkv, g, batch, n, heads, dim_head, scale, backward, out) -> None:
    check(load().bcosk_attention(_p(qkv), _p(g), batch, n, heads, dim_head, C.c_float(scale), int(backward), _p(out), _stream()),
          "bcosk_attention")


# ------------------------------------------------------------------------------------------------
# fine-tuning step (csrc/bcosk_train.cu, csrc/bcosk_wgrad.cu)
# ------------------------------------------------------------------------------------------------
def wgrad(p: "WgradParams") -> None:
    check(load().bcosk_wgrad(C.byref(p), _stream()), "bcosk_wgrad")


def bnu_stats_nhwc(x, rows, c, dtype, partials) -> None:
    """partials: [nblk, 2c] fp32 (one row per launched block, summed in order by bnu_finalize)"""
    check(load().bcosk_bnu_stats_nhwc(_p(x), C.c_int64(rows), c, dtype, _p(partials), partials.shape[0], _stream()), "bcosk_bnu_stats_nhwc")


def bnu_finalize(partials, rows, c, weight, eps, momentum, running_var, alpha, mean, rstd) -> None:
    check(load().bcosk_bnu_finalize(_p(partials), partials.shape[0], C.c_int64(rows), c, _p(weight), C.c_float(eps), C.c_float(momentum),
                                    _p(running_var), _p(alpha), _p(mean), _p(rstd), _stream()), "bcosk_bnu_finalize")


def bnu_apply_nhwc(x, rows, c, alpha, res, relu, y, sq, dtype) -> None:
    check(load().bcosk_bnu_apply_nhwc(_p(x), C.c_int64(rows), c, _p(alpha), _p(res), int(relu), _p(y), _p(sq), dtype, _stream()),
          "bcosk_bnu_apply_nhwc")


def train_bwd_reduce(ga, ga_f32, gb, xpost, tn, relu, out, out_f32, rows, c, partials, dtype) -> None:
    check(load().bcosk_train_bwd_reduce(_p(ga), int(ga_f32), _p(gb), _p(xpost), _p(tn), int(relu), _p(out), int(out_f32),
                                        C.c_int64(rows), c, _p(partials), partials.shape[0], dtype, _stream()), "bcosk_train_bwd_reduce")


def bnu_bwd_finalize(partials, rstd, weight, rows, c, kcoef, g_weight, s_out=None) -> None:
    check(load().bcosk_bnu_bwd_finalize(_p(partials), partials.shape[0], _p(rstd), _p(weight), C.c_int64(rows), c, _p(kcoef),
                                        _p(g_weight), _p(s_out), _stream()), "bcosk_bnu_bwd_finalize")


def train_bwd_apply(ga, ga_f32, gb, xpost, tn, relu, out, out_f32, scale, alpha, kcoef, mean, inv_norm, rows, c, g_lin, gnt, g_y,
                    dtype) -> None:
    check(load().bcosk_train_bwd_apply(_p(ga), int(ga_f32), _p(gb), _p(xpost), _p(tn), int(relu), _p(out), int(out_f32), _p(scale),
                                       _p(alpha), _p(kcoef), _p(mean), _p(inv_norm), C.c_int64(rows), c, _p(g_lin), _p(gnt), _p(g_y),
                                       dtype, _stream()), "bcosk_train_bwd_apply")


def grad_combine(ga, gb, x, tn, rows, c, out, dtype) -> None:
    check(load().bcosk_grad_combine(_p(ga), _p(gb), _p(x), _p(tn), C.c_int64(rows), c, _p(out), dtype, _stream()), "bcosk_grad_combine")


def pool_bwd_norm(ga, ga_f32, gb, xp, tn, nb, h, w, c, k, accumulate, gx, dtype) -> None:
    check(load().bcosk_pool_bwd_norm(_p(ga), int(ga_f32), _p(gb), _p(xp), _p(tn), nb, h, w, c, k, int(accumulate), _p(gx), dtype, _stream()),
          "bcosk_pool_bwd_norm")


def sumpool_transpose(gnt, nb, h, w, k, stride, pad, op, oq, accumulate, tn) -> None:
    check(load().bcosk_sumpool_transpose(_p(gnt), nb, h, w, k, stride, pad, op, oq, int(accumulate), _p(tn), _stream()),
          "bcosk_sumpool_transpose")


def bce_uniform_off(logits, labels, n, c, off_label, inv_temp, npix, grad_scale, loss, g_fc, g_logits, dtype) -> None:
    check(load().bcosk_bce_uniform_off(_p(logits), _p(labels), n, c, C.c_float(off_label), C.c_float(inv_temp), npix,
                                       C.c_float(grad_scale), _p(loss), _p(g_fc), _p(g_logits), dtype, _stream()),
          "bcosk_bce_uniform_off")


def gather_cast(src, idx, n, out, dtype) -> None:
    check(load().bcosk_gather_cast(_p(src), _p(idx), C.c_int64(n), _p(out), dtype, _stream()), "bcosk_gather_cast")


def adam_state_step(state, beta1, beta2) -> None:
    check(load().bcosk_adam_state_step(_p(state), C.c_float(beta1), C.c_float(beta2), _stream()), "bcosk_adam_state_step")


def agc_adamw_multi(w, g, gidx, m, v, unit_off, unit_cols, units, grad_scale, lr, beta1, beta2, eps, weight_decay, clip_factor, agc_eps,
                    adam_state) -> None:
    check(load().bcosk_agc_adamw_multi(_p(w), _p(g), _p(gidx), _p(m), _p(v), _p(unit_off), _p(unit_cols), units, C.c_float(grad_scale),
                                       C.c_float(lr), C.c_float(beta1), C.c_float(beta2), C.c_float(eps), C.c_float(weight_decay),
                                       C.c_float(clip_factor), C.c_float(agc_eps), _p(adam_state), _stream()), "bcosk_agc_adamw_multi")


def gather_cast_multi(src, table, npacks, max_n, dtype) -> None:
    check(load().bcosk_gather_cast_multi(_p(src), _p(table), npacks, C.c_int64(max_n), dtype, _stream()), "bcosk_gather_cast_multi")


def agc_adamw(w, g, gidx, m, v, units, cols, grad_scale, lr, beta1, beta2, eps, weight_decay, clip_factor, agc_eps, step) -> None:
    check(load().bcosk_agc_adamw(_p(w), _p(g), _p(gidx), _p(m), _p(v), units, cols, C.c_float(grad_scale), C.c_float(lr),
                                 C.c_float(beta1), C.c_float(beta2), C.c_float(eps), C.c_float(weight_decay), C.c_float(clip_factor),
                                 C.c_float(agc_eps), step, _stream()), "bcosk_agc_adamw")


# ---- DenseNet fine-tuning step (csrc/bcosk_dense_train.cu)
def dense_slice_stats(F, rows, ld, col0, c, eps, partials, mean, var, rstd, dtype) -> None:
    """partials: [nblk, 2c] fp32 scratch; mean / var / rstd: the block's [C_total] arrays, channels [col0, col0 + c) written"""
    check(load().bcosk_dense_slice_stats(_p(F), C.c_int64(rows), ld, col0, c, C.c_float(eps), _p(partials), partials.shape[0], _p(mean),
                                         _p(var), _p(rstd), dtype, _stream()), "bcosk_dense_slice_stats")


def dense_consumer_finalize(var, rstd, weight, c, momentum, running_var, alpha) -> None:
    check(load().bcosk_dense_consumer_finalize(_p(var), _p(rstd), _p(weight), c, C.c_float(momentum), _p(running_var), _p(alpha), _stream()),
          "bcosk_dense_consumer_finalize")


def dense_consumer_bwd(g_t, t, gnt, alpha, F, ld, rows, c, G, accumulate, partials, dtype) -> None:
    """partials: [nblk, c] fp32 (one row per launched block, summed in order by dense_consumer_bwd_finalize)"""
    import torch
    check(load().bcosk_dense_consumer_bwd(_p(g_t), int(g_t.dtype == torch.float32), _p(t), _p(gnt), _p(alpha), _p(F), ld, C.c_int64(rows), c,
                                          _p(G), int(accumulate), _p(partials), partials.shape[0], dtype, _stream()), "bcosk_dense_consumer_bwd")


def dense_consumer_bwd_finalize(partials, rstd, weight, rows, c, accumulate, K, g_weight) -> None:
    check(load().bcosk_dense_consumer_bwd_finalize(_p(partials), partials.shape[0], _p(rstd), _p(weight), C.c_int64(rows), c, int(accumulate),
                                                   _p(K), _p(g_weight), _stream()), "bcosk_dense_consumer_bwd_finalize")


def dense_slice_bwd(G, F, ld, col0, rows, c, mean, K, scale, inv_norm, out, gnt, dtype) -> None:
    check(load().bcosk_dense_slice_bwd(_p(G), _p(F), ld, col0, C.c_int64(rows), c, _p(mean), _p(K), _p(scale), _p(inv_norm), _p(out), _p(gnt),
                                       dtype, _stream()), "bcosk_dense_slice_bwd")
