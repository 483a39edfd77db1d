"""Tensor-level wrappers over the C ABI.  torch is used for device memory and streams only.

Activations are channels-last bf16 2-D/4-D tensors on a CUDA device; every wrapper validates device /
dtype / contiguity and raises (no CPU fallback -- a CPU tensor is an error, SURVEY.md section 8b).
"""
from __future__ import annotations

import torch

from . import _lib

ACT_DTYPE = torch.bfloat16   # storage dtype of activations / activation gradients in HBM
ACT = {None: 0, "none": 0, "relu": 1, "hswish": 2, "gelu": 3, "gelu_tanh": 4, "relu6": 5, "sigmoid": 6}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


# ------------------------------------------------------------------------------------ precision mode
# "bf16"  : bf16 operands / activations, fp32 accumulation on tcgen05 / mma.sync -- the fast path (3e-3 .. 1.5e-2 from fp32).
# "strict": fp32 activations, weights and FMA accumulation on the CUDA cores (csrc/strict_f32.cu) -- the parity mode for
#           north_star's tolerances (embeddings rtol 1e-4, mask logits rtol 1e-3, binary masks bit-exact).
_PRECISION = "bf16"


def precision() -> str:
    return _PRECISION


class strict_precision:
    """`with ops.strict_precision():` -- modules that implement the strict mode run it inside (EfficientViT students, SAM heads, FPN
    neck); the others raise rather than silently answering in bf16."""

    def __init__(self, enabled: bool = True):
        self.mode = "strict" if enabled else "bf16"

    def __enter__(self):
        global _PRECISION
        self.prev, _PRECISION = _PRECISION, self.mode
        return self

    def __exit__(self, *exc):
        global _PRECISION
        _PRECISION = self.prev


# ------------------------------------------------------------------------------------ accounting
# kernels launched per C-ABI call (memsets excluded) -- bench.py reports the sum as `gpu_launches`.
KERNELS_PER_CALL = {"es3_colsum_f32": 2, "es3_layernorm_bwd": 2, "es3_litemla_attn": 2, "es3_litemla_attn_generic": 2, "es3_fill_small_components": 4, "es3_grad_norm": 2, "es3_adamw_flat": 2, "es3_litemla_attn_tc": 2, "es3_kd_loss_fwd": 2, "es3_channel_mean": 2, "es3_preprocess_images": 2}
launch_count = 0


class Profiler:
    """Optional per-call CUDA-event timing with algorithmic bytes / flops (bench.py roofline leg).
    Events are recorded on the current stream, which is the stream the kernels are launched on."""

    def __init__(self):
        self.records = []  # (name, start_event, end_event, bytes, flops)

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1, nbytes, flops in self.records:
            a = agg.setdefault(name, dict(calls=0, ms=0.0, bytes=0, flops=0))
            a["calls"] += 1
            a["ms"] += e0.elapsed_time(e1)
            a["bytes"] += nbytes
            a["flops"] += flops
        return agg


_profiler: Profiler | None = None


def set_profiler(p: Profiler | None):
    global _profiler
    _profiler = p


def _nb(*ts):
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def _call(name, tag, nbytes, flops, *args):
    """Launch one C-ABI op; `tag` names the kernel family for the profiler."""
    global launch_count
    launch_count += KERNELS_PER_CALL.get(name, 1)
    if _profiler is None:
        _lib.call(name, *args)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    _lib.call(name, *args)
    e1.record()
    _profiler.records.append((tag, e0, e1, nbytes, flops))


def _chk(t: torch.Tensor, dtype, name: str):
    if not t.is_cuda:
        raise _lib.Es3Error(f"{name}: expected a CUDA tensor (the native path has no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.Es3Error(f"{name}: expected {dtype}, got {t.dtype}")
    return t


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _ensure_init(t: torch.Tensor):
    _lib.init(t.device.index or 0)


PW_SMALL = True    # K, N <= 64 plain pointwise GEMMs on es3_pw_small_bf16 (CUDA cores, HBM-bound) instead of 128-row tcgen05 tiles


def gemm(a, w, *, scale=None, bias=None, act=None, residual=None, out=None, out_dtype=torch.bfloat16, bn_hint=0,
         rope=None, act_after_res=False):
    """out[m,n] = act(scale[n]*sum_k a[m,k] w[n,k] + bias[n]) (+residual).  a: [M,K] (row stride allowed),
    w: [N,K] bf16, scale/bias fp32 [N]; residual bf16 or fp32 [M,N].
    rope = (table[P,32,2] fp32, rope_cols, H, W, win): rotate columns [0, rope_cols) (see es3_gemm_bf16_ex)."""
    _chk(a, torch.bfloat16, "a"); _chk(w, torch.bfloat16, "w")
    _ensure_init(a)
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K, (a.shape, w.shape)
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=out_dtype)
    assert out.stride(1) == 1 and out.shape == (M, N)
    res_f32 = 0
    if residual is not None:
        assert residual.is_cuda and residual.dtype in (torch.bfloat16, torch.float32)
        assert residual.stride(1) == 1 and residual.shape == (M, N)
        res_f32 = int(residual.dtype == torch.float32)
    if (PW_SMALL and K <= 64 and N <= 64 and scale is None and bias is None and act in (None, "none") and rope is None
            and out.dtype == torch.bfloat16 and (residual is None or residual.dtype == torch.bfloat16)):
        # 16..64-channel pointwise convs of stages 0-1 (and their input gradients): one thread per pixel row (pw_small.cu)
        global launch_count
        prof = _profiler
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        rc = _lib.call_rc("es3_pw_small_bf16", a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(), out.stride(0),
                          _ptr(residual), residual.stride(0) if residual is not None else 0, M, N, K, _stream())
        if rc == 0:
            launch_count += 1
            if prof is not None:
                e1.record()
                prof.records.append((f"pw_small[K={K},N={N}]", e0, e1, M * K * 2 + M * N * 2 + _nb(w, residual), 2 * M * N * K))
            return out
    if rope is not None:
        tab, rcols, rH, rW, rwin = rope
        _chk(tab, torch.float32, "rope table")
        assert tab.is_contiguous() and tab.shape[1:] == (32, 2)
        rargs = (tab.data_ptr(), rcols, rH, rW, rwin)
    else:
        rargs = (0, 0, 0, 0, 0)
    _call("es3_gemm_bf16_ex", f"gemm_tc[K={K},N={N}]", M * K * 2 + M * N * out.element_size() + _nb(w, residual),
          2 * M * N * K, a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), out.data_ptr(), out.stride(0),
          int(out.dtype == torch.float32), M, N, K, _ptr(scale), _ptr(bias), ACT[act], _ptr(residual),
          residual.stride(0) if residual is not None else 0, res_f32, *rargs, int(act_after_res), bn_hint, _stream())
    return out


def gemm_simt(a, w, *, scale=None, bias=None, act=None, residual=None, out=None, out_dtype=torch.bfloat16):
    _ensure_init(a)
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=out_dtype)
    res_f32 = int(residual is not None and residual.dtype == torch.float32)
    _call("es3_gemm_simt", "gemm_simt", _nb(a, w, out, residual), 2 * M * N * K, a.data_ptr(), a.stride(0), int(a.dtype == torch.float32), w.data_ptr(), w.stride(0),
              int(w.dtype == torch.float32), out.data_ptr(), out.stride(0), int(out.dtype == torch.float32), M, N, K,
              _ptr(scale), _ptr(bias), ACT[act], _ptr(residual), residual.stride(0) if residual is not None else 0,
              res_f32, _stream())
    return out


def conv3x3(x, w9, *, scale=None, bias=None, act=None, residual=None, out_dtype=torch.bfloat16, bn_hint=0):
    """x: [B,H,W,C] bf16 NHWC contiguous; w9: [N, 9*C] bf16 (tap-major k)."""
    _chk(x, torch.bfloat16, "x"); _chk(w9, torch.bfloat16, "w9")
    _ensure_init(x)
    assert x.is_contiguous() and w9.is_contiguous()
    B, H, W, Cc = x.shape
    N = w9.shape[0]
    assert w9.shape[1] == 9 * Cc
    out = torch.empty((B, H, W, N), device=x.device, dtype=out_dtype)
    _call("es3_conv3x3_bf16", f"conv3x3_tc[C={Cc},N={N}]", _nb(x, w9, out, residual), 2 * B * H * W * N * 9 * Cc,
          x.data_ptr(), w9.data_ptr(), out.data_ptr(), int(out_dtype == torch.float32),
              B, H, W, Cc, N, _ptr(scale), _ptr(bias), ACT[act], _ptr(residual), bn_hint, _stream())
    return out


def stem_conv3x3_s2(x, w27, bias, act):
    """x: [B,3,H,W] fp32 NCHW -> [B,Ho,Wo,Cout] bf16 NHWC.  w27: [27,Cout] fp32."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, _, H, W = x.shape
    Cout = w27.shape[1]
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
    _call("es3_stem_conv3x3_s2", "stem_conv3x3_s2", _nb(x, out), 2 * B * Ho * Wo * Cout * 27, x.data_ptr(), w27.data_ptr(), _ptr(bias), out.data_ptr(), B, H, W, Cout,
              ACT[act], _stream())
    return out


def round_taps_sum_bf16(w):
    """w [taps, C] fp32 -> fp32 tensor of bf16-representable taps whose per-channel sum stays (nearly) the fp32 sum."""
    _chk(w, torch.float32, "w")
    _ensure_init(w)
    assert w.dim() == 2 and w.is_contiguous() and w.shape[0] <= 25
    out = torch.empty_like(w)
    _call("es3_round_taps_sum_bf16", "round_taps", 2 * _nb(w), w.numel(), w.data_ptr(), out.data_ptr(), w.shape[0], w.shape[1], _stream())
    return out


def _tc_taps(w):
    """The tensor-core kernel's tap operand of `w`, computed once per (tensor object, version)."""
    c = getattr(w, "_es3_tc_taps", None)
    if c is None or c[0] != w._version:
        c = (w._version, round_taps_sum_bf16(w))
        w._es3_tc_taps = c
    return c[1]


DW_TC = True   # stride-1 3x3 / 5x5 depthwise convs with C % 32 == 0 on the tensor-core kernel (csrc/dw_tc.cu; GPU parity: test_dwconv_tc)


def dwconv(x, w, bias, ks, stride, act, out=None, force_simple=False, impl=None):
    """x: [B,H,W,C] bf16 (channel-sliced views allowed); w: [ks*ks, C] fp32.  impl: None (default routing), "tc" (tensor-core kernel,
    stride 1), "tiled" (CUDA-core shared-memory kernel)."""
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    B, H, W, Cc = x.shape
    assert x.stride(3) == 1 and x.stride(1) == W * x.stride(2) and x.stride(0) == H * x.stride(1)
    pad = ks // 2
    Ho, Wo = (H + 2 * pad - ks) // stride + 1, (W + 2 * pad - ks) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=torch.bfloat16)
    if DW_TC and stride == 1 and ks in (3, 5) and Cc % 32 == 0 and not force_simple and impl in (None, "tc"):
        _call("es3_dwconv_tc_bf16", f"dwconv_tc{ks}x{ks}", B * H * W * Cc * 2 + B * Ho * Wo * Cc * 2, 2 * B * Ho * Wo * Cc * ks * ks,
              x.data_ptr(), x.stride(2), _tc_taps(w).data_ptr(), _ptr(bias), out.data_ptr(), out.stride(2), B, H, W, Cc, ks, ACT[act], _stream())
        return out
    fn = "es3_dwconv_tiled_bf16" if (Cc % 32 == 0 and not force_simple) else "es3_dwconv_bf16"
    _call(fn, f"dwconv{ks}x{ks}s{stride}", B * H * W * Cc * 2 + B * Ho * Wo * Cc * 2, 2 * B * Ho * Wo * Cc * ks * ks,
          x.data_ptr(), x.stride(2), w.data_ptr(), _ptr(bias), out.data_ptr(), out.stride(2),
              B, H, W, Cc, ks, stride, ACT[act], _stream())
    return out


def dsconv_res(x, wdw, bdw, wpw, bpw, act):
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, Cc = x.shape
    out = torch.empty_like(x)
    _call("es3_dsconv_res_bf16", "dsconv_res", _nb(x, out), 2 * B * H * W * Cc * (9 + Cc), x.data_ptr(), wdw.data_ptr(), _ptr(bdw), wpw.data_ptr(), _ptr(bpw),
              out.data_ptr(), B, H, W, Cc, ACT[act], _stream())
    return out


def stem_fused_c16(x, w0, s0, b0, wdw, bdw, wpw, spw, bpw):
    """EfficientViT-B1 stem conv + DSConv residual in one launch.  x: [B,3,H,W] fp32 -> [B,Ho,Wo,16] bf16."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, _, H, W = x.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((B, Ho, Wo, 16), device=x.device, dtype=torch.bfloat16)
    _call("es3_stem_fused_c16", "stem_fused_c16", _nb(x, out), 2 * B * Ho * Wo * 16 * (27 + 9 + 16),
          x.data_ptr(), w0.data_ptr(), s0.data_ptr(), b0.data_ptr(), _tc_taps(wdw).data_ptr(), bdw.data_ptr(), wpw.data_ptr(),
          spw.data_ptr(), bpw.data_ptr(), out.data_ptr(), B, H, W, _stream())
    return out


def bilinear_nhwc_to_nchw(x, Ho, Wo):
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, Hi, Wi, Cc = x.shape
    out = torch.empty((B, Cc, Ho, Wo), device=x.device, dtype=torch.float32)
    _call("es3_bilinear_nhwc_to_nchw", "bilinear_nhwc_to_nchw", _nb(x, out), 8 * out.numel(), x.data_ptr(), out.data_ptr(), B, Hi, Wi, Cc, Ho, Wo, _stream())
    return out


def nhwc_to_nchw_f32(x):
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, Cc = x.shape
    out = torch.empty((B, Cc, H, W), device=x.device, dtype=torch.float32)
    _call("es3_nhwc_to_nchw_f32", "nhwc_to_nchw", _nb(x, out), 0, x.data_ptr(), out.data_ptr(), B, H * W, Cc, _stream())
    return out


def nchw_f32_to_nhwc(x):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, Cc, H, W = x.shape
    out = torch.empty((B, H, W, Cc), device=x.device, dtype=torch.bfloat16)
    _call("es3_nchw_f32_to_nhwc", "nchw_to_nhwc", _nb(x, out), 0, x.data_ptr(), out.data_ptr(), B, H * W, Cc, _stream())
    return out


def litemla_aggreg(ms, wdw, wpw, C3, force_simple=False):
    """ms: [B,H,W,2*C3] bf16; fills channels [C3, 2*C3) in place."""
    _chk(ms, torch.bfloat16, "ms")
    _ensure_init(ms)
    assert ms.is_contiguous()
    B, H, W, ld = ms.shape
    fn = "es3_litemla_aggreg_tiled" if (C3 % 64 == 0 and not force_simple) else "es3_litemla_aggreg"
    _call(fn, "litemla_aggreg", 2 * B * H * W * C3 * 2, 2 * B * H * W * C3 * (25 + 16), ms.data_ptr(), ld, wdw.data_ptr(), wpw.data_ptr(), B, H, W, C3, _stream())
    return ms


def litemla_wcomb(wdw, wpw):
    """Combined aggreg weights: wdw [25, C3] fp32 (tap-major), wpw [C3, 16] fp32 -> [C3/16, 25, 16, 16] bf16."""
    C3 = wpw.shape[0]
    G = C3 // 16
    d = wdw.t().reshape(G, 16, 25)                     # [g][i][tap]
    w = wpw.reshape(G, 16, 16)                         # [g][n][i]
    comb = w.unsqueeze(1) * d.permute(0, 2, 1).unsqueeze(2)   # [g][tap][n][i]
    return comb.to(torch.bfloat16).contiguous()


def litemla_aggreg_tc(ms, wcomb, C3):
    _chk(ms, torch.bfloat16, "ms"); _chk(wcomb, torch.bfloat16, "wcomb")
    _ensure_init(ms)
    assert ms.is_contiguous() and wcomb.is_contiguous() and wcomb.shape == (C3 // 16, 25, 16, 16)
    B, H, W, ld = ms.shape
    _call("es3_litemla_aggreg_tc", "litemla_aggreg_tc", 2 * B * H * W * C3 * 2, 2 * B * H * W * C3 * 400,
          ms.data_ptr(), ld, wcomb.data_ptr(), B, H, W, C3, _stream())
    return ms


def litemla_dwpw_weights(wdw, wpw):
    """wdw [25, C3] fp32 (tap-major), wpw [C3, 16] fp32 -> ([C3/16, 25, 16] bf16, [C3, 16] bf16) for es3_litemla_aggreg_dwpw."""
    C3 = wpw.shape[0]
    d = round_taps_sum_bf16(wdw.contiguous()).reshape(25, C3 // 16, 16).permute(1, 0, 2)      # bf16 taps with the fp32 tap sums
    return d.to(torch.bfloat16).contiguous(), wpw.to(torch.bfloat16).contiguous()


def litemla_aggreg_dwpw(ms, wd, wp, C3):
    _chk(ms, torch.bfloat16, "ms"); _chk(wd, torch.bfloat16, "wd"); _chk(wp, torch.bfloat16, "wp")
    _ensure_init(ms)
    assert ms.is_contiguous() and wd.is_contiguous() and wp.is_contiguous()
    assert wd.shape == (C3 // 16, 25, 16) and wp.shape == (C3, 16)
    B, H, W, ld = ms.shape
    _call("es3_litemla_aggreg_dwpw", "litemla_aggreg_dwpw", 2 * B * H * W * C3 * 2, 2 * B * H * W * C3 * (25 + 16),
          ms.data_ptr(), ld, wd.data_ptr(), wp.data_ptr(), B, H, W, C3, _stream())
    return ms


def litemla_attn(ms, heads2, eps=1e-15, tc=True, return_kv=False):
    """ms: [B,H,W,48*heads2] bf16 -> att [B,H,W,16*heads2] bf16.  return_kv: also return the workspace holding the
    [B][heads2][ceil(HW/512)][17][16] partial KV sums (es3_litemla_attn_bwd consumes it)."""
    _chk(ms, torch.bfloat16, "ms")
    _ensure_init(ms)
    assert ms.is_contiguous()
    B, H, W, ld = ms.shape
    att = torch.empty((B, H, W, 16 * heads2), device=ms.device, dtype=torch.bfloat16)
    kv = torch.empty((B * heads2 * ((H * W + 511) // 512) * 17 * 16,), device=ms.device, dtype=torch.float32)
    _call("es3_litemla_attn_tc" if tc else "es3_litemla_attn", "litemla_attn_tc" if tc else "litemla_attn", _nb(ms) * 2 // 3 + _nb(ms) // 3 + _nb(att), 2 * B * H * W * heads2 * 17 * 16 * 2,
          ms.data_ptr(), ld, kv.data_ptr(), att.data_ptr(), att.shape[3], B, H * W, heads2,
              float(eps), _stream())
    return (att, kv) if return_kv else att


def litemla_attn_generic(ms, heads2, dim, eps=1e-15, return_kv=False):
    """ReLU linear attention for head dim 16 | 32 (CUDA-core kernels).  ms: [B,H,W,3*dim*heads2] bf16 -> [B,H,W,dim*heads2].
    return_kv: also return the partial-KV workspace (es3_litemla_attn_bwd_generic consumes it)."""
    _chk(ms, torch.bfloat16, "ms")
    _ensure_init(ms)
    assert ms.is_contiguous() and ms.shape[3] == 3 * dim * heads2
    B, H, W, ld = ms.shape
    att = torch.empty((B, H, W, dim * heads2), device=ms.device, dtype=torch.bfloat16)
    kv = torch.empty((B * heads2 * ((H * W + 127) // 128) * (dim + 1) * dim,), device=ms.device, dtype=torch.float32)
    _call("es3_litemla_attn_generic", f"litemla_attn_generic[{dim}]", _nb(ms, att), 2 * B * H * W * heads2 * (dim + 1) * dim * 2,
          ms.data_ptr(), ld, kv.data_ptr(), att.data_ptr(), att.shape[3], B, H * W, heads2, dim, float(eps), _stream())
    return (att, kv) if return_kv else att


MBCONV_TC = True   # stride-1 residual blocks on the tcgen05 kernel (es3_mbconv_tc_bf16); False -> mma.sync kernel only


def mbconv_fused(x, w1, s1, b1, wdw, b2, w3, s3, b3, stride, residual, act, impl=None):
    """Fused MBConv (expand -> dw3x3 -> project [+x]); returns None when the shape is not instantiated.
    impl: None = tcgen05 kernel where it applies, else the mma.sync kernel; "tc" / "mma" force one (None if not instantiated)."""
    global launch_count
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, Cin = x.shape
    Mid, Cout = w1.shape[0], w3.shape[0]
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    y = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
    wdw = _tc_taps(wdw)     # the fused kernels multiply bf16 taps: per-channel tap sums kept (es3_round_taps_sum_bf16), cached on the tensor
    args = (x.data_ptr(), y.data_ptr(), w1.data_ptr(), s1.data_ptr(), b1.data_ptr(), wdw.data_ptr(), b2.data_ptr(),
            w3.data_ptr(), s3.data_ptr(), b3.data_ptr(), B, H, W, Cin, Mid, Cout, stride, int(residual), ACT[act],
            _stream())
    prof = _profiler
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    rc, tag = -1, "mbconv_tc"
    if impl == "tc" or (impl is None and MBCONV_TC):
        rc = _lib.call_rc("es3_mbconv_tc_bf16", *args)
        if rc < 0:
            rc = _lib.call_rc("es3_mbconv_tc_s2_bf16", *args)
    if rc < 0 and impl != "tc":
        rc, tag = _lib.call_rc("es3_mbconv_fused_bf16", *args), "mbconv_fused"
    if rc < 0:
        return None
    launch_count += 1
    if prof is not None:
        e1.record()
        flops = 2 * B * (H * W * Cin * Mid + Ho * Wo * Mid * (9 + Cout))
        prof.records.append((f"{tag}[{Cin}-{Mid}-{Cout},s{stride}]", e0, e1, _nb(x, y), flops))
    return y


def dwproj(mid, wdw, b2, w3, s3, b3, residual=None, act="hswish"):
    """act(dw3x3(mid) + b2) -> 1x1 projection -> s3 * . + b3 (+ residual) in one tcgen05 kernel; None if the shape is not
    instantiated (the caller then runs dwconv + gemm).  mid [B,H,W,Mid] bf16, w3 [Cout, Mid] bf16, residual [B,H,W,Cout]."""
    global launch_count
    _chk(mid, torch.bfloat16, "mid"); _chk(w3, torch.bfloat16, "w3")
    _ensure_init(mid)
    assert mid.is_contiguous() and w3.is_contiguous()
    B, H, W, Mid = mid.shape
    Cout = w3.shape[0]
    if residual is not None:
        _chk(residual, torch.bfloat16, "residual")
        assert residual.is_contiguous() and residual.shape == (B, H, W, Cout)
    y = torch.empty((B, H, W, Cout), device=mid.device, dtype=torch.bfloat16)
    prof = _profiler
    if prof is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = _lib.call_rc("es3_dwproj_tc_bf16", mid.data_ptr(), _tc_taps(wdw).data_ptr(), b2.data_ptr(), w3.data_ptr(), s3.data_ptr(),
                      b3.data_ptr(), _ptr(residual), y.data_ptr(), B, H, W, Mid, Cout, ACT[act], _stream())
    if rc < 0:
        return None
    launch_count += 1
    if prof is not None:
        e1.record()
        prof.records.append((f"dwproj_tc[{Mid}-{Cout}]", e0, e1, _nb(mid, y, residual), 2 * B * H * W * Mid * (9 + Cout)))
    return y


def layernorm(x, gamma, beta, eps=1e-5, *, pos=None, pos_size=0, H=0, W=0, out_bf16=True, out_f32=False):
    """x: [M, C] fp32 -> (bf16 [M,C] | None, fp32 [M,C] | None); optional tiled abs-pos add before the norm."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    yb = torch.empty((M, C), device=x.device, dtype=torch.bfloat16) if out_bf16 else None
    yf = torch.empty((M, C), device=x.device, dtype=torch.float32) if out_f32 else None
    _call("es3_layernorm_f32", "layernorm", _nb(x, yb, yf), 8 * M * C, x.data_ptr(), _ptr(pos), pos_size, H, W,
          gamma.data_ptr(), beta.data_ptr(), float(eps), _ptr(yb), _ptr(yf), M, C, _stream())
    return yb, yf


def im2col_patch(x, P, Kp):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, _, S, _ = x.shape
    n = (S // P) ** 2
    cols = torch.empty((B * n, Kp), device=x.device, dtype=torch.bfloat16)
    _call("es3_im2col_patch", "im2col_patch", _nb(x, cols), 0, x.data_ptr(), cols.data_ptr(), B, S, P, Kp, _stream())
    return cols


def attention(qkv, B, H, W, C, num_heads, win, scale, impl=None):
    """qkv: [B*H*W, 3C] bf16 -> [B*H*W, C] bf16.  impl: None (dispatch), "tc" (tcgen05), "mma" (mma.sync)."""
    _chk(qkv, torch.bfloat16, "qkv")
    _ensure_init(qkv)
    assert qkv.is_contiguous() and qkv.shape == (B * H * W, 3 * C)
    out = torch.empty((B * H * W, C), device=qkv.device, dtype=torch.bfloat16)
    L = win * win if win else H * W
    _call({None: "es3_attention_bf16", "tc": "es3_attention_tc_bf16", "mma": "es3_attention_mma_bf16"}[impl], f"attention[L={L}]", _nb(qkv, out), 4 * B * H * W * L * C, qkv.data_ptr(), out.data_ptr(),
          B, H, W, C, num_heads, win, float(scale), _stream())
    return out


def tokens_f32_to_nchw(x, B, H, W):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    C = x.shape[-1]
    out = torch.empty((B, C, H, W), device=x.device, dtype=torch.float32)
    _call("es3_tokens_f32_to_nchw", "tokens_to_nchw", _nb(x, out), 0, x.data_ptr(), out.data_ptr(), B, H * W, C, _stream())
    return out


def cast_f32_to_f16(x, out=None):
    """fp32 -> fp16 (RN) of a contiguous tensor; `out` may be a preallocated fp16 staging buffer of the same numel."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    assert out.is_cuda and out.dtype == torch.float16 and out.is_contiguous() and out.numel() == x.numel()
    _call("es3_cast_f32_to_f16", "cast_f32_f16", x.numel() * 6, 0, x.data_ptr(), out.data_ptr(), x.numel(), _stream())
    return out


def preprocess_images(table, affine, S, max_out, taps_floats, in_bytes, out=None):
    """Resize + normalise + pad a batch of decoded images into out [B,3,S,S] fp32 (es3_preprocess_images).  table [B,16] int64
    and affine [B,6] fp32 are CUDA tensors as stage1.transforms.build_table lays them out; `in_bytes` (the images' bytes) is
    for the profiler.  `out` may be a preallocated buffer (a loader rotating the inputs of a graphed encoder)."""
    _chk(table, torch.int64, "table"); _chk(affine, torch.float32, "affine")
    _ensure_init(table)
    B = table.shape[0]
    assert table.shape == (B, 16) and affine.shape == (B, 6) and table.is_contiguous() and affine.is_contiguous()
    if out is None:
        out = torch.empty((B, 3, S, S), device=table.device, dtype=torch.float32)
    _chk(out, torch.float32, "out")
    if tuple(out.shape) != (B, 3, S, S) or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous [{B},3,{S},{S}] fp32 tensor, got {tuple(out.shape)}")
    taps = torch.empty(max(int(taps_floats), 1), device=table.device, dtype=torch.float32)
    _call("es3_preprocess_images", "preprocess", int(in_bytes) + _nb(out), 0, table.data_ptr(), affine.data_ptr(), taps.data_ptr(),
          B, S, max_out, out.data_ptr(), _stream())
    return out


# ------------------------------------------------------------------------------------ SAM heads
def convt2x2(x, wt, bias4=None, act=None, residual=None, out_dtype=torch.bfloat16, act_after_res=False):
    """ConvTranspose2d(k=2,s=2) on NHWC: x [B,H,W,Cin] bf16, wt [4*Cout, Cin] bf16 -> [B,2H,2W,Cout]."""
    _chk(x, torch.bfloat16, "x"); _chk(wt, torch.bfloat16, "wt")
    _ensure_init(x)
    assert x.is_contiguous() and wt.is_contiguous()
    B, H, W, Cin = x.shape
    Cout = wt.shape[0] // 4
    out = torch.empty((B, 2 * H, 2 * W, Cout), device=x.device, dtype=out_dtype)
    res_f32 = int(residual is not None and residual.dtype == torch.float32)
    if residual is not None:
        assert residual.is_contiguous() and residual.shape == out.shape
    _call("es3_convt2x2_bf16", f"convt2x2[{Cin}->{Cout}]", _nb(x, wt, out, residual), 2 * B * H * W * Cin * 4 * Cout,
          x.data_ptr(), wt.data_ptr(), out.data_ptr(), int(out_dtype == torch.float32), B, H, W, Cin, Cout, _ptr(bias4),
          ACT[act], _ptr(residual), res_f32, int(act_after_res), _stream())
    return out


def convt2x2_weight(w):
    """nn.ConvTranspose2d weight [Cin,Cout,2,2] -> bf16 [4*Cout, Cin] with row (dy*2+dx)*Cout + co."""
    cin, cout = w.shape[:2]
    return w.detach().permute(2, 3, 1, 0).reshape(4 * cout, cin).to(torch.bfloat16).contiguous()


def dense_pe(gauss, h, w):
    _chk(gauss, torch.float32, "gauss")
    _ensure_init(gauss)
    F_ = gauss.shape[1]
    out = torch.empty((h * w, 2 * F_), device=gauss.device, dtype=torch.float32)
    _call("es3_dense_pe", "dense_pe", _nb(out), 0, gauss.contiguous().data_ptr(), F_, h, w, out.data_ptr(), _stream())
    return out


def point_embed(coords, labels, gauss, not_a_point, point_emb, img_w, img_h, pad=True):
    """coords [B,P,2] fp32, labels [B,P] int32 -> [B,P+pad,C] fp32 (pad: the padding point appended when no box is given)."""
    _chk(coords, torch.float32, "coords")
    _ensure_init(coords)
    B, P, _ = coords.shape
    F_ = gauss.shape[1]
    out = torch.empty((B, P + int(pad), 2 * F_), device=coords.device, dtype=torch.float32)
    _call("es3_point_embed", "point_embed", _nb(out), 0, coords.contiguous().data_ptr(),
          labels.to(torch.int32).contiguous().data_ptr(), gauss.contiguous().data_ptr(), not_a_point.contiguous().data_ptr(),
          point_emb.contiguous().data_ptr(), F_, B, P, int(pad), float(img_w), float(img_h), out.data_ptr(), _stream())
    return out


def mask_downscale_tokens(mask, weights, base=None, eps=1e-6, out_bf16=True, out_f32=True):
    """mask [B,1,4h,4w] fp32; weights = (w0,b0,g1,be1,w1,b1,g2,be2,w2,b2) fp32 contiguous -> token-major
    (bf16|None, fp32|None) [B*h*w, C] = base[row % base_rows] + mask_downscaling(mask)."""
    _chk(mask, torch.float32, "mask")
    _ensure_init(mask)
    mask = mask.contiguous()
    B, one, H4, W4 = mask.shape
    assert one == 1 and H4 % 4 == 0 and W4 % 4 == 0 and len(weights) == 10
    h, w = H4 // 4, W4 // 4
    C = weights[8].shape[0]
    for t in weights:
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
    if base is not None:
        _chk(base, torch.float32, "base")
        assert base.is_contiguous() and base.shape[1] == C
    yb = torch.empty((B * h * w, C), device=mask.device, dtype=torch.bfloat16) if out_bf16 else None
    yf = torch.empty((B * h * w, C), device=mask.device, dtype=torch.float32) if out_f32 else None
    _call("es3_mask_downscale_tokens", "mask_downscale", _nb(mask, yb, yf, base), 0, mask.data_ptr(), *[t.data_ptr() for t in weights],
          _ptr(base), base.shape[0] if base is not None else 0, _ptr(yf), _ptr(yb), B, h, w, C, float(eps), _stream())
    return yb, yf


def fill_small_components(masks, thr=0.0, max_hole_area=0.0, max_sprinkle_area=0.0):
    """masks [..., H, W] fp32 logits -> copy with small background holes / foreground sprinkles filled (8-connectivity)."""
    _chk(masks, torch.float32, "masks")
    _ensure_init(masks)
    x = masks.contiguous()
    H, W = x.shape[-2:]
    N = x.numel() // (H * W)
    out = torch.empty_like(x)
    ws = torch.empty((2, N * H * W), device=x.device, dtype=torch.int32)
    _call("es3_fill_small_components", "fill_small_components", _nb(x, out), 0, x.data_ptr(), out.data_ptr(), ws[0].data_ptr(),
          ws[1].data_ptr(), N, H, W, float(thr), float(max_hole_area), float(max_sprinkle_area), _stream())
    return out


def add_rows(x, add=None, out_bf16=False, out_f32=True):
    """x [M,C] fp32 + add [R,C] fp32 (row m % R) -> (bf16|None, fp32|None)."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    R = add.shape[0] if add is not None else 1
    if add is not None:
        assert add.is_contiguous() and add.shape[1] == C
    yb = torch.empty((M, C), device=x.device, dtype=torch.bfloat16) if out_bf16 else None
    yf = torch.empty((M, C), device=x.device, dtype=torch.float32) if out_f32 else None
    _call("es3_add_rows", "add_rows", _nb(x, yb, yf), M * C, x.data_ptr(), _ptr(add), M, C, R, _ptr(yb), _ptr(yf), _stream())
    return yb, yf


def nchw_to_tokens(x, addc=None, out_bf16=True, out_f32=True):
    """x [B,C,H,W] fp32 (+ per-channel addc) -> token-major ([B*HW,C] fp32 | None, bf16 | None)."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, C, H, W = x.shape
    yf = torch.empty((B * H * W, C), device=x.device, dtype=torch.float32) if out_f32 else None
    yb = torch.empty((B * H * W, C), device=x.device, dtype=torch.bfloat16) if out_bf16 else None
    _call("es3_nchw_f32_to_tokens", "nchw_to_tokens", _nb(x, yf, yb), 0, x.data_ptr(), _ptr(addc), _ptr(yf), _ptr(yb), B,
          H * W, C, _stream())
    return yf, yb


def attn_few_queries(q, k, v, heads, scale):
    """q [B,Tq,D] fp32; k,v [B,Tk,D] bf16 or fp32 -> [B,Tq,D] fp32."""
    _chk(q, torch.float32, "q")
    _ensure_init(q)
    B, Tq, D = q.shape
    Tk = k.shape[1]
    assert q.is_contiguous() and k.is_contiguous() and v.is_contiguous() and k.dtype == v.dtype
    out = torch.empty_like(q)
    _call("es3_attn_few_queries", f"attn_few_queries[Tk={Tk}]", _nb(q, k, v, out), 4 * B * Tq * Tk * D, q.data_ptr(), D,
          k.data_ptr(), v.data_ptr(), D, int(k.dtype == torch.float32), out.data_ptr(), D, B, heads, D // heads, Tq, Tk,
          float(scale), _stream())
    return out


def attn_few_keys(q, k, v, B, heads, scale):
    """q [B*Nq, D] bf16; k,v [B,Tk,D] fp32 -> [B*Nq, D] bf16."""
    _chk(q, torch.bfloat16, "q"); _chk(k, torch.float32, "k")
    _ensure_init(q)
    D = q.shape[1]
    Nq, Tk = q.shape[0] // B, k.shape[1]
    assert q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    out = torch.empty_like(q)
    _call("es3_attn_few_keys", "attn_few_keys", _nb(q, k, v, out), 4 * B * Nq * Tk * D, q.data_ptr(), D, k.data_ptr(),
          v.data_ptr(), D, out.data_ptr(), D, B, heads, D // heads, Nq, Tk, float(scale), _stream())
    return out


def ln_rows_gelu(x, w, b, eps):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    y = torch.empty((M, C), device=x.device, dtype=torch.bfloat16)
    _call("es3_ln_rows_gelu", "ln_rows_gelu", _nb(x, y), 10 * M * C, x.data_ptr(), w.data_ptr(), b.data_ptr(), float(eps),
          y.data_ptr(), M, C, _stream())
    return y


def hyper_masks(up, hyper, obj_logits, no_obj, K, k_off):
    """up [B,HW,32] fp32, hyper [B,Ktot,32] fp32 -> masks [B,K,HW] fp32 (object-gated when obj_logits given)."""
    _chk(up, torch.float32, "up"); _chk(hyper, torch.float32, "hyper")
    _ensure_init(up)
    assert up.is_contiguous() and hyper.is_contiguous()
    B, HW, CU = up.shape
    masks = torch.empty((B, K, HW), device=up.device, dtype=torch.float32)
    _call("es3_hyper_masks", "hyper_masks", _nb(up, masks), 2 * B * HW * K * CU, up.data_ptr(), hyper.data_ptr(),
          _ptr(obj_logits), float(no_obj), masks.data_ptr(), B, HW, CU, hyper.shape[1], K, k_off, _stream())
    return masks


def bilinear_nchw(x, Ho, Wo, binarize_thr=None, want_float=True):
    """x [B,C,Hi,Wi] fp32 -> (fp32 [B,C,Ho,Wo] | None, uint8 mask | None)."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    x = x.contiguous()
    B, C, Hi, Wi = x.shape
    out = torch.empty((B, C, Ho, Wo), device=x.device, dtype=torch.float32) if want_float else None
    binm = torch.empty((B, C, Ho, Wo), device=x.device, dtype=torch.uint8) if binarize_thr is not None else None
    _call("es3_bilinear_nchw_f32", "bilinear_nchw", _nb(x, out, binm), 8 * B * C * Ho * Wo, x.data_ptr(), _ptr(out), _ptr(binm),
          float(binarize_thr or 0.0), B * C, Hi, Wi, Ho, Wo, _stream())
    return out, binm


def maxpool2x2(x):
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, C = x.shape
    out = torch.empty((B, H // 2, W // 2, C), device=x.device, dtype=torch.bfloat16)
    _call("es3_maxpool2x2_bf16", "maxpool2x2", _nb(x, out), 0, x.data_ptr(), out.data_ptr(), B, H, W, C, _stream())
    return out


def kd_loss_fwd(preds, teacher, sizes_hw, img_size, cosine_weight):
    _chk(preds, torch.float32, "preds"); _chk(teacher, torch.float32, "teacher")
    _ensure_init(preds)
    preds, teacher = preds.contiguous(), teacher.contiguous()
    assert preds.shape == teacher.shape and preds.shape[-1] == preds.shape[-2]
    B, C, E, _ = preds.shape
    ws = torch.empty((B * ((E * E + 255) // 256) * 3,), device=preds.device, dtype=torch.float32)
    out = torch.empty((3,), device=preds.device, dtype=torch.float32)
    per = torch.empty((B, 3), device=preds.device, dtype=torch.float32)
    _call("es3_kd_loss_fwd", "kd_loss_fwd", _nb(preds, teacher), 8 * preds.numel(), preds.data_ptr(), teacher.data_ptr(),
          sizes_hw.contiguous().data_ptr(), B, C, E, img_size, float(cosine_weight), ws.data_ptr(), out.data_ptr(), per.data_ptr(),
          _stream())
    return out, per


def kd_loss_bwd(preds, teacher, sizes_hw, per_sample, img_size, cosine_weight, grad_scale=1.0, scale_dev=None):
    """Gradient of the KD loss w.r.t. preds ([B,C,E,E] fp32), times grad_scale (and the device loss scale scale_dev[0])."""
    _chk(preds, torch.float32, "preds"); _chk(teacher, torch.float32, "teacher")
    _ensure_init(preds)
    preds, teacher = preds.contiguous(), teacher.contiguous()
    B, C, E, _ = preds.shape
    out = torch.empty_like(preds)
    _call("es3_kd_loss_bwd", "kd_loss_bwd", 3 * _nb(preds), 8 * preds.numel(), preds.data_ptr(), teacher.data_ptr(),
          sizes_hw.contiguous().data_ptr(), per_sample.data_ptr(), _ptr(scale_dev), float(grad_scale), B, C, E, img_size,
          float(cosine_weight), out.data_ptr(), _stream())
    return out


def grad_norm(flat_grad, part_ws, norm_ws):
    """norm_ws[0] = sum g^2, norm_ws[1] = non-finite flag over the flat fp32 arena (no host sync)."""
    _chk(flat_grad, torch.float32, "flat_grad")
    _ensure_init(flat_grad)
    assert flat_grad.is_contiguous() and part_ws.numel() >= 8192 and norm_ws.numel() >= 2
    _call("es3_grad_norm", "grad_norm", _nb(flat_grad), 2 * flat_grad.numel(), flat_grad.data_ptr(), flat_grad.numel(),
          part_ws.data_ptr(), norm_ws.data_ptr(), _stream())


def adamw_flat(p, g, m, v, n_decay, lr, betas, eps, weight_decay, max_norm, inv_world, norm_ws, state, dynamic_scale=False,
               growth=2.0, backoff=0.5, growth_interval=2000):
    """Fused AdamW over flat arenas (see es3_adamw_flat in include/es3.h)."""
    for t in (p, g, m, v):
        _chk(t, torch.float32, "arena")
        assert t.is_contiguous() and t.numel() == p.numel()
    _ensure_init(p)
    _call("es3_adamw_flat", "adamw_flat", 7 * _nb(p), 12 * p.numel(), p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(),
          p.numel(), int(n_decay), float(lr), float(betas[0]), float(betas[1]), float(eps), float(weight_decay), float(max_norm),
          float(inv_world), norm_ws.data_ptr(), state.data_ptr(), int(dynamic_scale), float(growth), float(backoff),
          int(growth_interval), _stream())


def conv3x3_s2_narrow(x, w9, scale, bias, act=None):
    """x [B,H,W,Cin] bf16, w9 [9, Cout, Cin] bf16 -> [B,Ho,Wo,Cout] bf16 (dense 3x3, stride 2, pad 1, folded BN)."""
    _chk(x, torch.bfloat16, "x"); _chk(w9, torch.bfloat16, "w9")
    _ensure_init(x)
    assert x.is_contiguous() and w9.is_contiguous() and x.shape[3] == w9.shape[2]
    B, H, W, Cin = x.shape
    Cout = w9.shape[1]
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    out = torch.empty((B, Ho, Wo, Cout), device=x.device, dtype=torch.bfloat16)
    _call("es3_conv3x3_s2_narrow_bf16", f"conv3x3_s2[{Cin}-{Cout}]", _nb(x, out), 2 * B * Ho * Wo * Cout * 9 * Cin, x.data_ptr(),
          w9.data_ptr(), scale.data_ptr(), bias.data_ptr(), out.data_ptr(), B, H, W, Cin, Cout, ACT[act], _stream())
    return out


def channel_mean(x):
    """x [B,H,W,C] bf16 -> [B,C] fp32."""
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, C = x.shape
    ws = torch.empty((B * ((H * W + 127) // 128) * C,), device=x.device, dtype=torch.float32)
    mean = torch.empty((B, C), device=x.device, dtype=torch.float32)
    _call("es3_channel_mean", "channel_mean", _nb(x), B * H * W * C, x.data_ptr(), ws.data_ptr(), mean.data_ptr(), B, H * W, C, _stream())
    return mean


def scale_channels(x, gate):
    _chk(x, torch.bfloat16, "x"); _chk(gate, torch.float32, "gate")
    _ensure_init(x)
    assert x.is_contiguous() and gate.is_contiguous()
    B, H, W, C = x.shape
    y = torch.empty_like(x)
    _call("es3_scale_channels", "scale_channels", 2 * _nb(x), B * H * W * C, x.data_ptr(), gate.data_ptr(), y.data_ptr(), B, H * W, C, _stream())
    return y


def layernorm_bf16(x, gamma, beta, eps=1e-5):
    """x [M,C] bf16 -> bf16 (C % 8 == 0)."""
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    y = torch.empty_like(x)
    _call("es3_layernorm_bf16", "layernorm_bf16", 2 * _nb(x), 8 * M * C, x.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
          float(eps), y.data_ptr(), M, C, _stream())
    return y


def win_attn_bias(qkv, qkv_pad, bias, B, H, W, C, heads, ws, scale):
    """qkv [B*H*W, 3C] bf16 (per-head q|k|v blocks of 32), qkv_pad [3C] bf16, bias [heads, ws^2, ws^2] fp32."""
    _chk(qkv, torch.bfloat16, "qkv"); _chk(qkv_pad, torch.bfloat16, "qkv_pad"); _chk(bias, torch.float32, "bias")
    _ensure_init(qkv)
    assert qkv.is_contiguous() and bias.is_contiguous() and qkv.shape == (B * H * W, 3 * C)
    out = torch.empty((B * H * W, C), device=qkv.device, dtype=torch.bfloat16)
    _call("es3_win_attn_bias_bf16", f"win_attn_bias[ws={ws}]", _nb(qkv, out), 4 * B * H * W * ws * ws * C, qkv.data_ptr(),
          qkv_pad.data_ptr(), bias.data_ptr(), out.data_ptr(), B, H, W, C, heads, ws, float(scale), _stream())
    return out


# ------------------------------------------------------------------------------------ student backward (train_bwd.cu)
BN_MODE = {"none": 0, "eval": 1, "batch": 2}
KERNELS_PER_CALL.update({"es3_bn_stats": 2, "es3_bn_act_bwd_reduce": 2, "es3_wgrad_pw": 2, "es3_dwconv_wgrad": 2,
                         "es3_stem_wgrad": 2, "es3_litemla_attn_bwd": 4, "es3_dwconv_wgrad_tiled": 2, "es3_se_bwd_dgate": 2,
                         "es3_litemla_attn_bwd_generic": 2})


def _f32ws(n, dev):
    return torch.empty((max(int(n), 1),), device=dev, dtype=torch.float32)


def bn_stats(z, gamma, beta, eps, momentum, running_mean=None, running_var=None, num_batches_tracked=None):
    """Train-mode BatchNorm statistics of z [M,C] bf16 (any leading dims, C last, contiguous).
    Returns (mean, invstd, scale, shift) fp32 [C]; updates the running buffers in place (nn.BatchNorm2d semantics)."""
    _chk(z, torch.bfloat16, "z")
    _ensure_init(z)
    assert z.is_contiguous()
    C = z.shape[-1]
    M = z.numel() // C
    dev = z.device
    mean, invstd, scale, shift = (torch.empty(C, device=dev, dtype=torch.float32) for _ in range(4))
    ws = _f32ws(_lib.size("es3_col_reduce_ws_floats", M, C), dev)
    for t in (running_mean, running_var):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous())
    assert num_batches_tracked is None or num_batches_tracked.dtype == torch.int64
    _call("es3_bn_stats", "bn_stats", _nb(z), 3 * z.numel(), z.data_ptr(), M, C, float(eps), float(momentum), _ptr(gamma),
          _ptr(beta), ws.data_ptr(), mean.data_ptr(), invstd.data_ptr(), scale.data_ptr(), shift.data_ptr(),
          _ptr(running_mean), _ptr(running_var), _ptr(num_batches_tracked), _stream())
    return mean, invstd, scale, shift


def affine_act(z, scale, shift, act, residual=None, out=None):
    """act(scale[c] z + shift[c]) (+ residual) on [..., C] bf16 contiguous (out: optional contiguous destination of z's shape)."""
    _chk(z, torch.bfloat16, "z")
    _ensure_init(z)
    assert z.is_contiguous() and (residual is None or (residual.is_contiguous() and residual.shape == z.shape))
    C = z.shape[-1]
    if out is None:
        out = torch.empty_like(z)
    assert out.is_contiguous() and out.shape == z.shape and out.dtype == z.dtype
    _call("es3_affine_act", "affine_act", _nb(z, out, residual), 4 * z.numel(), z.data_ptr(), _ptr(scale), _ptr(shift), ACT[act],
          _ptr(residual), out.data_ptr(), z.numel() // C, C, _stream())
    return out


def bn_act_bwd(da, z, scale, shift, act, mode, mean=None, invstd=None, dgamma=None, dbeta=None, apply=True):
    """Backward through act(scale z + shift) and the norm that produced (scale, shift); see es3_bn_act_bwd_reduce.
    da, z: [..., C] bf16 contiguous.  dgamma / dbeta: fp32 [C] accumulated in place (None: not needed).  Returns dz bf16
    (apply=False: only the per-channel reductions, returns None)."""
    _chk(da, torch.bfloat16, "da"); _chk(z, torch.bfloat16, "z")
    _ensure_init(z)
    assert da.is_contiguous() and z.is_contiguous() and da.shape == z.shape
    C = z.shape[-1]
    M = z.numel() // C
    dev = z.device
    ws = _f32ws(_lib.size("es3_col_reduce_ws_floats", M, C), dev)
    coef = torch.empty((3, C), device=dev, dtype=torch.float32)
    _call("es3_bn_act_bwd_reduce", "bn_act_bwd_reduce", _nb(da, z), 6 * z.numel(), da.data_ptr(), z.data_ptr(), _ptr(scale),
          _ptr(shift), ACT[act], BN_MODE[mode], _ptr(mean), _ptr(invstd), M, C, ws.data_ptr(), coef.data_ptr(), _ptr(dgamma),
          _ptr(dbeta), _stream())
    if not apply:
        return None
    dz = torch.empty_like(z)
    _call("es3_bn_act_bwd_apply", "bn_act_bwd_apply", _nb(da, z, dz), 8 * z.numel(), da.data_ptr(), z.data_ptr(), _ptr(scale),
          _ptr(shift), ACT[act], coef.data_ptr(), dz.data_ptr(), M, C, _stream())
    return dz


def add_bf16(a, b):
    """a + b for 2-D bf16 matrices with unit column stride (row-strided views allowed) -> contiguous bf16."""
    _chk(a, torch.bfloat16, "a"); _chk(b, torch.bfloat16, "b")
    _ensure_init(a)
    assert a.dim() == 2 and a.shape == b.shape and a.stride(1) == 1 and b.stride(1) == 1
    M, C = a.shape
    out = torch.empty((M, C), device=a.device, dtype=torch.bfloat16)
    _call("es3_add_bf16", "add_bf16", 3 * M * C * 2, M * C, a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(),
          out.stride(0), M, C, _stream())
    return out


WGRAD_TC = True    # 1x1-conv weight gradients with N % 64 == 0 and K % 64 == 0 on the tcgen05 split-K kernel (es3_wgrad_tc)


def wgrad_pw(dz, x, dW, ldn=None, ldk=1, shift=None):
    """dW[n*ldn + k*ldk] += sum_m dz[m,n] x[m,k].  dz [M,N], x [M,K] bf16 (row strides allowed); dW fp32 (flat indexing
    from its data pointer).  shift = (H, W, dy, dx): x row of pixel (b,y,x) is (b,y+dy,x+dx), zero outside the map."""
    _chk(dz, torch.bfloat16, "dz"); _chk(x, torch.bfloat16, "x"); _chk(dW, torch.float32, "dW")
    _ensure_init(dz)
    assert dz.dim() == 2 and x.dim() == 2 and dz.stride(1) == 1 and x.stride(1) == 1 and dz.shape[0] == x.shape[0]
    M, N = dz.shape
    K = x.shape[1]
    if WGRAD_TC and shift is None and ldk == 1 and N % 64 == 0 and K % 64 == 0 and M >= 64:
        # dense contraction over the pixel index: split-K UMMA with both operands MN-major (wgrad_tc.cu)
        global launch_count
        ws = _f32ws(_lib.size("es3_wgrad_tc_ws_floats", M, N, K), dz.device)
        prof = _profiler
        if prof is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        rc = _lib.call_rc("es3_wgrad_tc", dz.data_ptr(), dz.stride(0), x.data_ptr(), x.stride(0), M, N, K, ws.data_ptr(), dW.data_ptr(),
                          K if ldn is None else ldn, _stream())
        if rc == 0:
            launch_count += 2
            if prof is not None:
                e1.record()
                prof.records.append((f"wgrad_tc[N={N},K={K}]", e0, e1, M * (N + K) * 2, 2 * M * N * K))
            return dW
    H, W, dy, dx = shift if shift is not None else (0, 0, 0, 0)
    ws = _f32ws(_lib.size("es3_wgrad_pw_ws_floats", M, N, K), dz.device)
    _call("es3_wgrad_pw", f"wgrad_pw[N={N},K={K}]", M * (N + K) * 2, 2 * M * N * K, dz.data_ptr(), dz.stride(0), x.data_ptr(),
          x.stride(0), M, N, K, H, W, dy, dx, ws.data_ptr(), dW.data_ptr(), K if ldn is None else ldn, ldk, _stream())
    return dW


def transpose_pad(x, Wp, dx):
    """x [B,H,W,C] bf16 -> [C, B*(H+2)*Wp] bf16: zero-framed, x-shifted transpose (es3_transpose_pad_bf16)."""
    _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, H, W, C = x.shape
    out = torch.empty((C, B * (H + 2) * Wp), device=x.device, dtype=torch.bfloat16)
    _call("es3_transpose_pad_bf16", "transpose_pad", _nb(x) + 2 * _nb(out), 0, x.data_ptr(), out.data_ptr(), B, H, W, C, Wp, dx, _stream())
    return out


def accumulate_strided(src, dst, inner, ld_outer, ld_inner):
    """dst.flat[(i // inner) * ld_outer + (i % inner) * ld_inner] += src.flat[i]  (fp32)."""
    _chk(src, torch.float32, "src"); _chk(dst, torch.float32, "dst")
    _ensure_init(src)
    assert src.is_contiguous()
    _call("es3_accumulate_strided", "accumulate_strided", 3 * _nb(src), src.numel(), src.data_ptr(), src.numel(), inner, ld_outer,
          ld_inner, dst.data_ptr(), _stream())
    return dst


def conv3x3_wgrad(dy, a, gw):
    """gw [N,C,3,3] fp32 += weight gradient of a dense 3x3 / pad 1 conv; dy [B,H,W,N], a [B,H,W,C] bf16 NHWC.
    Nine tcgen05 GEMMs over the zero-framed pixel index (see es3_transpose_pad_bf16 in include/es3.h)."""
    B, H, W, N = dy.shape
    C = a.shape[3]
    Wp = (W + 2 + 7) // 8 * 8
    Mp = B * (H + 2) * Wp
    dyT = transpose_pad(dy, Wp, 0)
    full = torch.empty((N, C), device=dy.device, dtype=torch.float32)
    flat = gw.view(-1)
    for kx in range(3):
        aT = transpose_pad(a, Wp, kx - 1)
        for ky in range(3):
            lo = Wp + (ky - 1) * Wp
            # 64-wide tiles: 8 x 16 = 128 CTAs instead of 64 on 148 SMs (the contraction runs over ~43 K pixels: MMA-bound per tile)
            gemm(dyT[:, Wp:Mp - Wp], aT[:, lo:lo + Mp - 2 * Wp], out=full, bn_hint=64 if full.shape[1] >= 512 else 0)
            accumulate_strided(full, flat[ky * 3 + kx:], C, 9 * C, 9)
    return gw


def dwconv_bwd_data(dz, w, H, W, ks, stride):
    """Input gradient of a depthwise conv (pad ks//2): dz [B,Ho,Wo,C] bf16, w [ks*ks, C] fp32 -> dx [B,H,W,C] bf16."""
    _chk(dz, torch.bfloat16, "dz"); _chk(w, torch.float32, "w")
    _ensure_init(dz)
    assert dz.is_contiguous() and w.is_contiguous()
    B, Ho, Wo, C = dz.shape
    pad = ks // 2
    assert Ho == (H + 2 * pad - ks) // stride + 1 and Wo == (W + 2 * pad - ks) // stride + 1
    dx = torch.empty((B, H, W, C), device=dz.device, dtype=torch.bfloat16)
    _call("es3_dwconv_bwd_data", f"dwconv_bwd_data{ks}x{ks}s{stride}", _nb(dz, dx), 2 * dz.numel() * ks * ks, dz.data_ptr(),
          w.data_ptr(), dx.data_ptr(), B, H, W, C, ks, stride, _stream())
    return dx


DW_WGRAD_WIN = True      # route C % 32 == 0 weight gradients (stride 1 | 2) to es3_dwconv_wgrad_win (GPU parity: test_dwconv_wgrad_win)
DW_WGRAD_TILED = True    # route stride-1, C % 32 == 0 weight gradients to es3_dwconv_wgrad_tiled (GPU parity: test_dwconv_wgrad_tiled, r2)


def dwconv_wgrad(dz, x, dW, ks, stride, impl=None):
    """dW [C,1,ks,ks] fp32 += depthwise weight gradient; dz [B,Ho,Wo,C] bf16 contiguous, x [B,H,W,C] bf16 (channel slice ok).
    impl="win": register sliding window over shared-memory tiles (C % 32 == 0; the default for such shapes); impl="tiled": the first
    shared-memory tiled kernel (stride 1, C % 32 == 0); impl="direct": the global-memory kernels."""
    _chk(dz, torch.bfloat16, "dz"); _chk(x, torch.bfloat16, "x"); _chk(dW, torch.float32, "dW")
    _ensure_init(dz)
    B, H, W, C = x.shape
    assert dz.is_contiguous() and dW.is_contiguous() and dW.numel() == C * ks * ks and dz.shape[3] == C
    assert x.stride(3) == 1 and x.stride(1) == W * x.stride(2) and x.stride(0) == H * x.stride(1)
    if impl == "win" or (impl is None and DW_WGRAD_WIN and C % 32 == 0):
        assert C % 32 == 0
        ws = _f32ws(_lib.size("es3_dwconv_wgrad_win_ws_floats", B, H, W, C, ks, stride), dz.device)
        _call("es3_dwconv_wgrad_win", f"dwconv_wgrad_win{ks}x{ks}s{stride}", _nb(dz) + B * H * W * C * 2, 2 * dz.numel() * ks * ks,
              dz.data_ptr(), x.data_ptr(), x.stride(2), B, H, W, C, ks, stride, ws.data_ptr(), dW.data_ptr(), _stream())
        return dW
    if impl == "tiled" or (impl is None and DW_WGRAD_TILED and stride == 1 and C % 32 == 0):   # (impl="direct" falls through)
        assert stride == 1 and C % 32 == 0
        ws = _f32ws(_lib.size("es3_dwconv_wgrad_tiled_ws_floats", B, H, W, C, ks), dz.device)
        _call("es3_dwconv_wgrad_tiled", f"dwconv_wgrad_tiled{ks}x{ks}", _nb(dz) + B * H * W * C * 2, 2 * dz.numel() * ks * ks,
              dz.data_ptr(), x.data_ptr(), x.stride(2), B, H, W, C, ks, ws.data_ptr(), dW.data_ptr(), _stream())
        return dW
    ws = _f32ws(_lib.size("es3_dwconv_wgrad_ws_floats", B, H, W, C, ks, stride), dz.device)
    _call("es3_dwconv_wgrad", f"dwconv_wgrad{ks}x{ks}s{stride}", _nb(dz) + B * H * W * C * 2, 2 * dz.numel() * ks * ks,
          dz.data_ptr(), x.data_ptr(), x.stride(2), B, H, W, C, ks, stride, ws.data_ptr(), dW.data_ptr(), _stream())
    return dW


def litemla_attn_bwd_generic(ms, datt, kv, heads2, dim, eps=1e-15):
    """Backward of litemla_attn_generic (head dim 16 | 32): ms [B,H,W,3*dim*heads2], datt [B,H,W,dim*heads2] bf16 -> dms like ms."""
    _chk(ms, torch.bfloat16, "ms"); _chk(datt, torch.bfloat16, "datt"); _chk(kv, torch.float32, "kv")
    _ensure_init(ms)
    assert ms.is_contiguous() and datt.is_contiguous() and ms.shape[3] == 3 * dim * heads2 and datt.shape[3] == dim * heads2
    B, H, W, ld = ms.shape
    HW = H * W
    dms = torch.empty_like(ms)
    ws = _f32ws(_lib.size("es3_litemla_bwd_generic_ws_floats", B, HW, heads2, dim), ms.device)
    _call("es3_litemla_attn_bwd_generic", f"litemla_attn_bwd_generic[{dim}]", 2 * _nb(ms, datt) + _nb(dms),
          2 * B * HW * heads2 * (dim + 1) * dim * 5, ms.data_ptr(), ld, datt.data_ptr(), datt.shape[3], kv.data_ptr(), (HW + 127) // 128,
          ws.data_ptr(), dms.data_ptr(), ld, B, HW, heads2, dim, float(eps), _stream())
    return dms


def layernorm_bwd(x, dy, gamma, eps, dgamma=None, dbeta=None, dres=None):
    """nn.LayerNorm backward over rows: x, dy [M,C] bf16 (the LN input and the gradient of its output) -> dx bf16 (+ dres);
    dgamma / dbeta fp32 [C] accumulated in place."""
    _chk(x, torch.bfloat16, "x"); _chk(dy, torch.bfloat16, "dy")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous() and dy.is_contiguous() and dy.shape == x.shape
    assert dres is None or (dres.is_contiguous() and dres.shape == x.shape and dres.dtype == x.dtype)
    M, C = x.shape
    dx = torch.empty_like(x)
    ws = _f32ws(_lib.size("es3_layernorm_bwd_ws_floats", M, C), x.device)
    _call("es3_layernorm_bwd", "layernorm_bwd", _nb(x, dy, dx, dres), 12 * x.numel(), x.data_ptr(), dy.data_ptr(), gamma.data_ptr(),
          _ptr(dres), float(eps), dx.data_ptr(), M, C, ws.data_ptr(), _ptr(dgamma), _ptr(dbeta), _stream())
    return dx


def win_attn_bias_bwd(qkv, dout, bias, B, H, W, C, heads, ws, scale):
    """Backward of win_attn_bias on a map with H, W multiples of ws: qkv [B*H*W, 3C], dout [B*H*W, C] bf16, bias [heads,N,N] fp32
    -> (dqkv [B*H*W, 3C] bf16, dbias [heads,N,N] fp32).  The kernel writes the per-window score gradients in fp32; their sum over the
    windows (the bias gradient) is es3_colsum_f32."""
    _chk(qkv, torch.bfloat16, "qkv"); _chk(dout, torch.bfloat16, "dout"); _chk(bias, torch.float32, "bias")
    _ensure_init(qkv)
    assert qkv.is_contiguous() and dout.is_contiguous() and bias.is_contiguous()
    assert qkv.shape == (B * H * W, 3 * C) and dout.shape == (B * H * W, C) and H % ws == 0 and W % ws == 0
    N = ws * ws
    nwin = B * (H // ws) * (W // ws)
    row = heads * N * N
    dS = torch.empty((nwin, row), device=qkv.device, dtype=torch.float32)
    dqkv = torch.empty_like(qkv)
    _call("es3_win_attn_bias_bwd", f"win_attn_bias_bwd[ws={ws}]", 2 * _nb(qkv) + _nb(dout, dS), 16 * B * H * W * N * C, qkv.data_ptr(),
          dout.data_ptr(), bias.data_ptr(), dqkv.data_ptr(), dS.data_ptr(), row, B, H, W, C, heads, ws, float(scale), _stream())
    dbias = torch.zeros(row, device=qkv.device, dtype=torch.float32)
    colsum_f32(dS, dbias)                                                        # fp32 sum over the windows, fixed order
    return dqkv, dbias.view(heads, N, N)


def colsum_f32(src, out):
    """out[c] += sum_r src[r, c] for an fp32 matrix (unit column stride), deterministic two-stage reduction."""
    _chk(src, torch.float32, "src"); _chk(out, torch.float32, "out")
    _ensure_init(src)
    assert src.dim() == 2 and src.stride(1) == 1 and out.is_contiguous() and out.numel() == src.shape[1]
    M, L = src.shape
    ws = _f32ws(_lib.size("es3_colsum_f32_ws_floats", M, L), src.device)
    _call("es3_colsum_f32", "colsum_f32", _nb(src), M * L, src.data_ptr(), src.stride(0), M, L, ws.data_ptr(), out.data_ptr(), _stream())
    return out


SE_BWD_BATCHED = True    # SqueezeExcite backward through es3_se_bwd_* instead of per-image loops (GPU parity: test_se_bwd_batched, r2)


def se_bwd_dgate(dy, x):
    """dgate [B,C] fp32 = sum over pixels of dy * x; dy, x [B,H,W,C] bf16 contiguous."""
    _chk(dy, torch.bfloat16, "dy"); _chk(x, torch.bfloat16, "x")
    _ensure_init(x)
    assert dy.is_contiguous() and x.is_contiguous() and dy.shape == x.shape
    B, H, W, C = x.shape
    dgate = torch.zeros((B, C), device=x.device, dtype=torch.float32)
    ws = _f32ws(_lib.size("es3_se_bwd_ws_floats", B, H * W, C), x.device)
    _call("es3_se_bwd_dgate", "se_bwd_dgate", _nb(dy, x), 2 * x.numel(), dy.data_ptr(), x.data_ptr(), B, H * W, C, ws.data_ptr(),
          dgate.data_ptr(), _stream())
    return dgate


def se_bwd_apply(dy, gate, add):
    """dy * gate[b,c] + add[b,c]; dy [B,H,W,C] bf16, gate / add [B,C] fp32 -> bf16."""
    _chk(dy, torch.bfloat16, "dy"); _chk(gate, torch.float32, "gate"); _chk(add, torch.float32, "add")
    _ensure_init(dy)
    assert dy.is_contiguous() and gate.is_contiguous() and add.is_contiguous()
    B, H, W, C = dy.shape
    dx = torch.empty_like(dy)
    _call("es3_se_bwd_apply", "se_bwd_apply", 2 * _nb(dy), 2 * dy.numel(), dy.data_ptr(), gate.data_ptr(), add.data_ptr(), dx.data_ptr(),
          B, H * W, C, _stream())
    return dx


def stem_wgrad(img, dz, dW):
    """dW [Cout,3,3,3] fp32 += weight gradient of the 3x3 stride-2 stem conv; img [B,3,H,W] fp32, dz [B,Ho,Wo,Cout] bf16."""
    _chk(img, torch.float32, "img"); _chk(dz, torch.bfloat16, "dz"); _chk(dW, torch.float32, "dW")
    _ensure_init(dz)
    img = img.contiguous()
    B, _, H, W = img.shape
    Cout = dz.shape[3]
    assert dz.is_contiguous() and dW.is_contiguous() and dW.numel() == Cout * 27
    ws = _f32ws(_lib.size("es3_stem_wgrad_ws_floats", B, H, W, Cout), dz.device)
    _call("es3_stem_wgrad", "stem_wgrad", _nb(img, dz), 2 * dz.numel() * 27, img.data_ptr(), dz.data_ptr(), B, H, W, Cout,
          ws.data_ptr(), dW.data_ptr(), _stream())
    return dW


def bilinear_bwd(dout, Hi, Wi):
    """Adjoint of bilinear_nhwc_to_nchw: dout [B,C,Ho,Wo] fp32 -> [B,Hi,Wi,C] bf16."""
    _chk(dout, torch.float32, "dout")
    _ensure_init(dout)
    dout = dout.contiguous()
    B, C, Ho, Wo = dout.shape
    din = torch.empty((B, Hi, Wi, C), device=dout.device, dtype=torch.bfloat16)
    _call("es3_bilinear_bwd", "bilinear_bwd", _nb(dout, din), 8 * dout.numel(), dout.data_ptr(), din.data_ptr(), B, Hi, Wi, C, Ho, Wo,
          _stream())
    return din


def litemla_attn_bwd(ms, datt, kv, heads2, eps=1e-15):
    """Backward of litemla_attn (head dim 16).  ms [B,H,W,48*heads2] bf16, datt [B,H,W,16*heads2] bf16, kv: the workspace
    litemla_attn(..., return_kv=True) returned.  Returns dms [B,H,W,48*heads2] bf16."""
    _chk(ms, torch.bfloat16, "ms"); _chk(datt, torch.bfloat16, "datt"); _chk(kv, torch.float32, "kv")
    _ensure_init(ms)
    assert ms.is_contiguous() and datt.is_contiguous()
    B, H, W, ld = ms.shape
    HW = H * W
    dms = torch.empty_like(ms)
    ws = _f32ws(_lib.size("es3_litemla_bwd_ws_floats", B, HW, heads2), ms.device)
    _call("es3_litemla_attn_bwd", "litemla_attn_bwd", 2 * _nb(ms, datt) + _nb(dms), 2 * B * HW * heads2 * 17 * 16 * 5,
          ms.data_ptr(), ld, datt.data_ptr(), datt.shape[3], kv.data_ptr(), (HW + 511) // 512, ws.data_ptr(), dms.data_ptr(), ld,
          B, HW, heads2, float(eps), _stream())
    return dms


# ------------------------------------------------------------------------------------ strict (fp32-class) mode ops (strict_f32.cu)
def sgemm(a, w, *, scale=None, bias=None, act=None, residual=None, out=None, act_after_res=False):
    """fp32 out[m,n] = act(scale[n] * sum_k a[m,k] w[n,k] + bias[n]) (+ residual); row strides allowed, unit column stride."""
    _chk(a, torch.float32, "a"); _chk(w, torch.float32, "w")
    _ensure_init(a)
    assert a.dim() == 2 and w.dim() == 2 and a.stride(1) == 1 and w.stride(1) == 1 and a.shape[1] == w.shape[1], (a.shape, w.shape)
    M, K = a.shape
    N = w.shape[0]
    if out is None:
        out = torch.empty((M, N), device=a.device, dtype=torch.float32)
    assert out.dtype == torch.float32 and out.shape == (M, N) and out.stride(1) == 1
    if residual is not None:
        _chk(residual, torch.float32, "residual")
        assert residual.shape == (M, N) and residual.stride(1) == 1
    _call("es3_sgemm_f32", f"sgemm_f32[K={K},N={N}]", 4 * (M * K + M * N) + _nb(w, residual), 2 * M * N * K, a.data_ptr(), a.stride(0),
          w.data_ptr(), w.stride(0), out.data_ptr(), out.stride(0), M, N, K, _ptr(scale), _ptr(bias), ACT[act], _ptr(residual),
          residual.stride(0) if residual is not None else 0, int(act_after_res), _stream())
    return out


def conv2d_f32(x, weight, stride=1, pad=0, *, scale=None, bias=None, act=None, residual=None, nchw=False):
    """Dense nn.Conv2d in the strict mode: x NHWC fp32 [B,H,W,C] (nchw=True: the NCHW fp32 image), weight [N,C,k,k] fp32 (the
    nn.Conv2d parameter) -> NHWC fp32 [B,Ho,Wo,N] = act(scale * conv + bias) (+ residual).  1x1 stride-1 convs are one SGEMM on the
    pixel matrix; everything else goes through es3_im2col_f32."""
    _chk(x, torch.float32, "x"); _chk(weight, torch.float32, "weight")
    _ensure_init(x)
    N, C, ks, _ = weight.shape
    if nchw:
        B, Cx, H, W = x.shape
    else:
        B, H, W, Cx = x.shape
    assert Cx == C and x.is_contiguous(), (x.shape, weight.shape)
    Ho, Wo = (H + 2 * pad - ks) // stride + 1, (W + 2 * pad - ks) // stride + 1
    res2 = residual.reshape(B * Ho * Wo, N) if residual is not None else None
    if ks == 1 and stride == 1 and pad == 0 and not nchw:
        out = sgemm(x.view(-1, C), weight.reshape(N, C), scale=scale, bias=bias, act=act, residual=res2)
        return out.view(B, Ho, Wo, N)
    cols = torch.empty((B * Ho * Wo, ks * ks * C), device=x.device, dtype=torch.float32)
    _call("es3_im2col_f32", "im2col_f32", _nb(x, cols), 0, x.data_ptr(), cols.data_ptr(), B, H, W, C, ks, stride, pad, int(nchw), _stream())
    wk = weight.permute(0, 2, 3, 1).reshape(N, ks * ks * C).contiguous()          # k = (ky * ks + kx) * C + c
    return sgemm(cols, wk, scale=scale, bias=bias, act=act, residual=res2).view(B, Ho, Wo, N)


def dwconv_f32(x, w, scale, bias, ks, stride, act, out=None):
    """Depthwise conv in the strict mode: x [B,H,W,C] fp32 (channel slice of a wider NHWC map allowed), w [ks*ks, C] fp32."""
    _chk(x, torch.float32, "x"); _chk(w, torch.float32, "w")
    _ensure_init(x)
    B, H, W, C = x.shape
    assert x.stride(3) == 1 and x.stride(1) == W * x.stride(2) and x.stride(0) == H * x.stride(1) and w.shape == (ks * ks, C) and w.is_contiguous()
    pad = ks // 2
    Ho, Wo = (H + 2 * pad - ks) // stride + 1, (W + 2 * pad - ks) // stride + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, C), device=x.device, dtype=torch.float32)
    assert out.shape == (B, Ho, Wo, C) and out.stride(3) == 1 and out.stride(1) == Wo * out.stride(2) and out.stride(0) == Ho * out.stride(1)
    _call("es3_dwconv_f32", f"dwconv_f32[k={ks}]", 4 * (x.numel() + out.numel()), 2 * out.numel() * ks * ks, x.data_ptr(), x.stride(2),
          w.data_ptr(), _ptr(scale), _ptr(bias), out.data_ptr(), out.stride(2), B, H, W, C, ks, stride, ACT[act], _stream())
    return out


def litemla_attn_f32(ms, heads, dim, eps):
    """LiteMLA.relu_linear_att on fp32: ms [B,H,W,3*dim*heads] (head = q | k | v) -> [B,H,W,dim*heads] fp32."""
    _chk(ms, torch.float32, "ms")
    _ensure_init(ms)
    assert ms.is_contiguous()
    B, H, W, ld = ms.shape
    assert ld == 3 * dim * heads
    out = torch.empty((B, H, W, dim * heads), device=ms.device, dtype=torch.float32)
    ws = _f32ws(_lib.size("es3_litemla_attn_f32_ws_floats", B, H * W, heads, dim), ms.device)
    _call("es3_litemla_attn_f32", "litemla_attn_f32", _nb(ms, out) + _nb(ms) * 2 // 3, 4 * B * H * W * heads * dim * (dim + 1),
          ms.data_ptr(), ld, ws.data_ptr(), out.data_ptr(), dim * heads, B, H * W, heads, dim, float(eps), _stream())
    return out


def bilinear_nhwc_f32_to_nchw(x, Ho, Wo):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.is_contiguous()
    B, Hi, Wi, C = x.shape
    out = torch.empty((B, C, Ho, Wo), device=x.device, dtype=torch.float32)
    _call("es3_bilinear_nhwc_f32_to_nchw", "bilinear_f32", _nb(x, out), 8 * out.numel(), x.data_ptr(), out.data_ptr(), B, Hi, Wi, C, Ho, Wo,
          _stream())
    return out


def attn_few_keys_f32(q, k, v, B, heads, scale):
    """q [B*Nq, D] fp32; k, v [B,Tk,D] fp32 -> [B*Nq, D] fp32 (libm exp)."""
    _chk(q, torch.float32, "q"); _chk(k, torch.float32, "k"); _chk(v, torch.float32, "v")
    _ensure_init(q)
    D = q.shape[1]
    Nq, Tk = q.shape[0] // B, k.shape[1]
    assert q.is_contiguous() and k.is_contiguous() and v.is_contiguous()
    out = torch.empty_like(q)
    _call("es3_attn_few_keys_f32", "attn_few_keys_f32", _nb(q, k, v, out), 4 * B * Nq * Tk * D, q.data_ptr(), D, k.data_ptr(), v.data_ptr(),
          D, out.data_ptr(), D, B, heads, D // heads, Nq, Tk, float(scale), _stream())
    return out


def ln_rows_gelu_f32(x, w, b, eps):
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    y = torch.empty_like(x)
    _call("es3_ln_rows_gelu_f32", "ln_rows_gelu_f32", 2 * _nb(x), 10 * M * C, x.data_ptr(), w.data_ptr(), b.data_ptr(), float(eps),
          y.data_ptr(), M, C, _stream())
    return y


def bias_act_res_f32(x, bias=None, act=None, residual=None, act_after_res=False):
    """act(x + bias[c]) + residual (act_after_res: act(x + bias[c] + residual)); x [..., C] fp32 contiguous."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.is_contiguous() and (residual is None or (residual.is_contiguous() and residual.shape == x.shape and residual.dtype == torch.float32))
    y = torch.empty_like(x)
    _call("es3_bias_act_res_f32", "bias_act_res_f32", _nb(x, y, residual), x.numel(), x.data_ptr(), _ptr(bias), _ptr(residual), y.data_ptr(),
          x.numel(), x.shape[-1], ACT[act], int(act_after_res), _stream())
    return y


def convt2x2_f32(x, weight, bias=None, act=None, residual=None, act_after_res=False):
    """nn.ConvTranspose2d(k=2, s=2) in the strict mode: x [B,H,W,Cin] fp32, weight [Cin,Cout,2,2] fp32 (the parameter) ->
    [B,2H,2W,Cout] fp32 = act(convT + bias) (+ residual).  One SGEMM with N = 4 Cout, depth-to-space as a view permute (layout
    plumbing), then the elementwise tail."""
    _chk(x, torch.float32, "x"); _chk(weight, torch.float32, "weight")
    B, H, W, Cin = x.shape
    Cout = weight.shape[1]
    wt = weight.permute(2, 3, 1, 0).reshape(4 * Cout, Cin).contiguous()          # row (dy*2+dx)*Cout + co
    y = sgemm(x.reshape(-1, Cin), wt)                                            # [B*H*W, 4*Cout]
    y = y.view(B, H, W, 2, 2, Cout).permute(0, 1, 3, 2, 4, 5).reshape(B, 2 * H, 2 * W, Cout).contiguous()
    return bias_act_res_f32(y, bias, act, residual, act_after_res)


def ln_rows_f32(x, w, b, eps):
    """nn.LayerNorm over the rows of an fp32 matrix of any width."""
    _chk(x, torch.float32, "x")
    _ensure_init(x)
    assert x.dim() == 2 and x.is_contiguous()
    M, C = x.shape
    y = torch.empty_like(x)
    _call("es3_ln_rows_f32", "ln_rows_f32", 2 * _nb(x), 8 * M * C, x.data_ptr(), w.data_ptr(), b.data_ptr(), float(eps), y.data_ptr(), M, C,
          _stream())
    return y


def rope_f32(qkv, table, rope_cols, H, W, win):
    """In-place 2-D axial RoPE on columns [0, rope_cols) of fp32 rows; table [positions, 32, 2] fp32 (cos, sin)."""
    _chk(qkv, torch.float32, "qkv"); _chk(table, torch.float32, "table")
    _ensure_init(qkv)
    assert qkv.dim() == 2 and qkv.stride(1) == 1 and table.is_contiguous() and table.shape[1:] == (32, 2)
    _call("es3_rope_f32", "rope_f32", 2 * qkv.shape[0] * rope_cols * 4, 6 * qkv.shape[0] * rope_cols // 2, qkv.data_ptr(), qkv.stride(0),
          qkv.shape[0], table.data_ptr(), rope_cols, H, W, win, _stream())
    return qkv


def attention_f32(qkv, B, H, W, heads, head_dim, win, scale, *, layout="blocks", bias=None, pad_row=None):
    """fp32 softmax attention over token rows qkv [B*H*W, ld] fp32 -> [B*H*W, heads*head_dim] fp32.  layout "blocks": q | k | v column
    blocks of heads*head_dim (the ViT trunk); "per_head": (q, k, v) triples per head (TinyViT).  win = 0: global; bias [heads, L, L];
    pad_row [ld] stands in for the tokens an overhanging window lacks."""
    _chk(qkv, torch.float32, "qkv")
    _ensure_init(qkv)
    C = heads * head_dim
    assert qkv.is_contiguous() and qkv.shape == (B * H * W, 3 * C), (qkv.shape, B, H, W, C)
    offs = (0, C, 2 * C, head_dim) if layout == "blocks" else (0, head_dim, 2 * head_dim, 3 * head_dim)
    L = win * win if win else H * W
    if bias is not None:
        _chk(bias, torch.float32, "bias")
        assert bias.is_contiguous() and bias.shape == (heads, L, L)
    if pad_row is not None:
        _chk(pad_row, torch.float32, "pad_row")
        assert pad_row.is_contiguous() and pad_row.numel() == 3 * C
    out = torch.empty((B * H * W, C), device=qkv.device, dtype=torch.float32)
    _call("es3_attention_f32", f"attention_f32[L={L}]", _nb(qkv, out), 4 * B * H * W * L * C, qkv.data_ptr(), out.data_ptr(), _ptr(bias),
          _ptr(pad_row), B, H, W, 3 * C, heads, head_dim, *offs, win, float(scale), _stream())
    return out


def scale_channels_f32(x, gate):
    """x [B,H,W,C] fp32 * gate [B,C] fp32."""
    _chk(x, torch.float32, "x"); _chk(gate, torch.float32, "gate")
    _ensure_init(x)
    assert x.is_contiguous() and gate.is_contiguous()
    B, H, W, C = x.shape
    y = torch.empty_like(x)
    _call("es3_scale_channels_f32", "scale_channels_f32", 2 * _nb(x), x.numel(), x.data_ptr(), gate.data_ptr(), y.data_ptr(), B, H * W, C,
          _stream())
    return y
