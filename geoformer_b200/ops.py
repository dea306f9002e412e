"""Torch-tensor front end of the C ABI (include/geoformer_b200.h).

Every function here launches hand-written sm_100a kernels from libgeoformer_sm100.so on the
current CUDA stream.  PyTorch is used for device memory and streams only.
"""
from __future__ import annotations

import os
import threading
from typing import Optional, Tuple

import torch

from . import _lib

EPI_RELU, EPI_TANH, EPI_ELU1, EPI_LN = 1, 2, 4, 8

# 'tf32' -> tcgen05 kind::tf32 tensor-core path (product default); 'ref' -> fp32 FFMA kernels
# (accuracy mode for parity runs; same ABI contract).  Both are sm_100a CUDA from this library.
_LINEAR_IMPL = "tf32"
_SIM_IMPL = "f16x3"
_ATTN_IMPL = "tf32"
# fp16 storage of the intermediates that only feed MMAs (which round to a 10-bit mantissa anyway) or the linear
# attention kernels: projected Q/K/V, attention message, MLP hidden.  The residual stream stays fp32.
_ACT16 = os.environ.get("GF_ACT16", "1") != "0"


def act16() -> bool:
    return _ACT16 and _LINEAR_IMPL == "tf32"


def set_precision(linear: Optional[str] = None, similarity: Optional[str] = None,
                  attention: Optional[str] = None, activations: Optional[str] = None) -> None:
    global _LINEAR_IMPL, _SIM_IMPL, _ATTN_IMPL, _ACT16
    if activations is not None:
        assert activations in ("f16", "f32")
        _ACT16 = activations == "f16"
    if attention is not None:
        assert attention in ("tf32", "tf32_mat", "ref")
        _ATTN_IMPL = attention
    if linear is not None:
        assert linear in ("tf32", "ref")
        _LINEAR_IMPL = linear
    if similarity is not None:
        assert similarity in ("f16x3", "ref")
        _SIM_IMPL = similarity


_PRECISION_LOCK = threading.RLock()


class precision_scope:
    """`with precision_scope(linear=..., similarity=..., attention=..., activations=...)`: run a block under its own
    precision options and restore the module-level ones afterwards.  The options are process-wide, so the scope holds a
    lock for its whole duration: blocks with an override run one at a time (GeoFormer.precision uses this; the default,
    no override, takes no lock and keeps MatchPipeline's batches concurrent)."""

    def __init__(self, **opts):
        self.opts = opts

    def __enter__(self):
        _PRECISION_LOCK.acquire()
        self.saved = (_LINEAR_IMPL, _SIM_IMPL, _ATTN_IMPL, _ACT16)
        set_precision(**self.opts)
        return self

    def __exit__(self, *exc):
        global _LINEAR_IMPL, _SIM_IMPL, _ATTN_IMPL, _ACT16
        _LINEAR_IMPL, _SIM_IMPL, _ATTN_IMPL, _ACT16 = self.saved
        _PRECISION_LOCK.release()
        return False


class _Profile:
    """Optional instrumentation: CUDA-event timing of regions on the launching stream (bench.py --stage-times) and /
    or NVTX ranges around every stage and C-ABI call (GF_NVTX=1, or PROFILE.nvtx = True) so that a timeline profiler
    names them.  Both are off by default and cost one attribute test per call when off."""

    def __init__(self):
        self.pattern = None
        self.records = {}
        self.nvtx = os.environ.get("GF_NVTX", "0") == "1"

    def enable(self, pattern: str) -> None:
        self.pattern, self.records = pattern, {}

    def disable(self) -> None:
        self.pattern = None

    def on(self, name: str) -> bool:
        return self.pattern is not None and (self.pattern == "*" or self.pattern in name)

    class _Region:
        def __init__(self, prof, name):
            self.prof, self.name = prof, name

        def __enter__(self):
            self.pushed = self.prof.nvtx
            if self.pushed:
                torch.cuda.nvtx.range_push(self.name)
            if self.prof.on(self.name):
                self.e0 = torch.cuda.Event(enable_timing=True)
                self.e1 = torch.cuda.Event(enable_timing=True)
                self.e0.record()
            else:
                self.e0 = None
            return self

        def __exit__(self, *exc):
            if self.e0 is not None:
                self.e1.record()
                self.prof.records.setdefault(self.name, []).append((self.e0, self.e1))
            if self.pushed:
                torch.cuda.nvtx.range_pop()
            return False

    def region(self, name: str):
        return _Profile._Region(self, name)

    def collect(self, name: str):
        torch.cuda.synchronize()
        return [a.elapsed_time(b) for k, v in self.records.items() if name in k for a, b in v]

    def summary(self):
        torch.cuda.synchronize()
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in self.records.items()}


PROFILE = _Profile()


def _call(name: str, *args, tag: str = "") -> None:
    """Launch through the C ABI, optionally timed as region 'k:<name><tag>'."""
    if PROFILE.pattern is None and not PROFILE.nvtx:
        _lib.call(name, *args)
    else:
        with PROFILE.region("k:" + name[3:] + tag):
            _lib.call(name, *args)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _chk(t: torch.Tensor, dtype=torch.float32) -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.GeoFormerLibError("geoformer_b200 ops need CUDA tensors (no CPU fallback)")
    assert t.dtype == dtype, (t.dtype, dtype)
    return t


def ensure_init(device: torch.device) -> None:
    idx = device.index if device.index is not None else torch.cuda.current_device()
    _lib.init(idx)


def linear(a: torch.Tensor, w: torch.Tensor, a2: Optional[torch.Tensor] = None, epi: int = 0, act_cols: int = 0,
           bias: Optional[torch.Tensor] = None, rowbias: Optional[torch.Tensor] = None, rowbias_group: int = 0,
           gamma: Optional[torch.Tensor] = None, beta: Optional[torch.Tensor] = None,
           residual: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None,
           impl: Optional[str] = None, out_f16: bool = False) -> torch.Tensor:
    """y[M,N] = epilogue([a | a2] @ w.T); a [M,K1], a2 [M,K2] (optional), w [N,K1+K2], all contiguous fp32 — or all
    fp16 (kind::f16 MMA, tensor-core path only).  out_f16: fp16 result (lean epilogue: no LN / residual / row bias)."""
    in_f16 = a.dtype == torch.float16
    if in_f16 or out_f16:
        return _linear_mixed(a, w, a2, epi, act_cols, bias, rowbias, rowbias_group, gamma, beta, residual, in_f16, out_f16, out)
    _chk(a); _chk(w)
    m, k1 = a.shape
    n = w.shape[0]
    k2 = 0 if a2 is None else a2.shape[1]
    assert a.is_contiguous() and w.is_contiguous() and w.shape[1] == k1 + k2
    if a2 is not None:
        assert a2.is_contiguous() and a2.shape[0] == m
    if residual is not None:
        assert residual.is_contiguous() and residual.shape == (m, n)
    y = out if out is not None else torch.empty((m, n), device=a.device, dtype=torch.float32)
    fn = "gf_linear_tf32" if (impl or _LINEAR_IMPL) == "tf32" else "gf_linear_ref"
    _call(fn, a.data_ptr(), _ptr(a2), w.data_ptr(), y.data_ptr(), m, n, k1, k2, epi, act_cols, _ptr(bias),
          _ptr(rowbias), rowbias_group, _ptr(gamma), _ptr(beta), _ptr(residual), None, _stream(),
          tag=f"[{n}x{k1 + k2}]")
    return y


def _linear_mixed(a, w, a2, epi, act_cols, bias, rowbias, rowbias_group, gamma, beta, residual, in_f16, out_f16, out=None):
    dt = torch.float16 if in_f16 else torch.float32
    _chk(a, dt); _chk(w, dt)
    if (_LINEAR_IMPL != "tf32"):
        raise _lib.GeoFormerLibError("fp16 activations exist on the tensor-core path only (set_precision(linear='tf32'))")
    m, k1 = a.shape
    n = w.shape[0]
    k2 = 0 if a2 is None else a2.shape[1]
    assert a.is_contiguous() and w.is_contiguous() and w.shape[1] == k1 + k2
    if a2 is not None:
        _chk(a2, dt)
        assert a2.is_contiguous() and a2.shape[0] == m
    if residual is not None:
        assert residual.is_contiguous() and residual.shape == (m, n) and residual.dtype == torch.float32
    ydt = torch.float16 if out_f16 else torch.float32
    if out is not None:
        assert out.shape == (m, n) and out.dtype == ydt and out.is_contiguous()
    y = out if out is not None else torch.empty((m, n), device=a.device, dtype=ydt)
    _call("gf_linear_mixed", a.data_ptr(), _ptr(a2), w.data_ptr(), y.data_ptr(), int(in_f16), int(out_f16), m, n, k1, k2,
          epi, act_cols, _ptr(bias), _ptr(rowbias), rowbias_group, _ptr(gamma), _ptr(beta), _ptr(residual), None,
          _stream(), tag=f"[{n}x{k1 + k2}{'h' if in_f16 else ''}{'>h' if out_f16 else ''}]")
    return y


def conv3x3(x: torch.Tensor, wt: torch.Tensor, bias: torch.Tensor, residual: Optional[torch.Tensor] = None,
            act: int = 0) -> torch.Tensor:
    """3x3/s1/p1 conv + folded BN (+ residual) + activation on NHWC fp16 (tcgen05 implicit GEMM).
    x [b,h,w,cin_p]; wt [cout_p, 9, cin_k]; bias fp32 [cout_p]; returns [b,h,w,cout_p] fp16."""
    return conv(x, wt, bias, residual, act, 1)


def conv(x: torch.Tensor, wt: torch.Tensor, bias: torch.Tensor, residual: Optional[torch.Tensor] = None,
         act: int = 0, stride: int = 1) -> torch.Tensor:
    """3x3 (pad 1) or 1x1 (pad 0) conv, stride 1 or 2, + bias (+ residual) + activation on NHWC fp16.
    wt [cout_p, taps, cin_k] with taps in {9, 1}; returns [b, (h-1)//stride+1, (w-1)//stride+1, cout_p] fp16."""
    assert x.dtype == torch.float16 and x.is_contiguous() and wt.dtype == torch.float16 and wt.is_contiguous()
    b, h, w, cin_p = x.shape
    cout_p, taps, cin_k = wt.shape
    assert taps in (1, 9)
    y = torch.empty((b, (h - 1) // stride + 1, (w - 1) // stride + 1, cout_p), device=x.device, dtype=torch.float16)
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous() and residual.dtype == torch.float16
    _call("gf_conv_f16", x.data_ptr(), wt.data_ptr(), bias.data_ptr(), _ptr(residual), y.data_ptr(), b, h, w, cin_p,
          cout_p, cin_k, 3 if taps == 9 else 1, stride, act, _stream(),
          tag=f"[{cin_p}->{cout_p}@{h}x{w}{'k1' if taps == 1 else ''}{'s2' if stride == 2 else ''}]")
    return y


def stem_conv(img: torch.Tensor, wperm: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """7x7/s2 stem + folded BN + ReLU: fp32 [b,1,h,w] -> NHWC fp16 [b,h/2,w/2,128]."""
    assert img.dtype == torch.float32 and img.is_contiguous() and img.shape[1] == 1
    b, _, h, w = img.shape
    out = torch.empty((b, (h - 1) // 2 + 1, (w - 1) // 2 + 1, 128), device=img.device, dtype=torch.float16)
    _call("gf_stem_conv7x7_f16", img.data_ptr(), wperm.data_ptr(), bias.data_ptr(), out.data_ptr(), b, h, w, _stream())
    return out


def upsample_add(lateral: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """lateral [b,h,w,c] + bilinear_upsample(src [b,hs,ws,c]) (align_corners=True), NHWC fp16."""
    assert lateral.is_contiguous() and src.is_contiguous() and lateral.dtype == src.dtype == torch.float16
    b, h, w, c = lateral.shape
    out = torch.empty_like(lateral)
    _call("gf_upsample_add_f16", lateral.data_ptr(), src.data_ptr(), out.data_ptr(), b, h, w, src.shape[1], src.shape[2],
          c, _stream())
    return out


def conv_ref(x: torch.Tensor, wt: torch.Tensor, bias: Optional[torch.Tensor], residual: Optional[torch.Tensor] = None,
             act: int = 0, stride: int = 1) -> torch.Tensor:
    """fp32 FFMA convolution (accurate mode): x NHWC fp32 [b,h,w,cin]; wt [k*k, cin, cout] fp32; pad = k // 2."""
    _chk(x); _chk(wt)
    assert x.is_contiguous() and wt.is_contiguous()
    b, h, w, cin = x.shape
    taps, cin_w, cout = wt.shape
    k = {1: 1, 9: 3, 49: 7}[taps]
    assert cin_w == cin
    pad = k // 2
    y = torch.empty((b, (h + 2 * pad - k) // stride + 1, (w + 2 * pad - k) // stride + 1, cout), device=x.device)
    if residual is not None:
        assert residual.shape == y.shape and residual.is_contiguous() and residual.dtype == torch.float32
    _call("gf_conv_ref", x.data_ptr(), wt.data_ptr(), _ptr(bias), _ptr(residual), y.data_ptr(), b, h, w, cin, cout, k,
          stride, act, _stream(), tag=f"[{cin}->{cout}@{h}x{w}k{k}s{stride}]")
    return y


def upsample_add_ref(lateral: torch.Tensor, src: torch.Tensor) -> torch.Tensor:
    """fp32 version of upsample_add (accurate mode)."""
    _chk(lateral); _chk(src)
    assert lateral.is_contiguous() and src.is_contiguous()
    b, h, w, c = lateral.shape
    out = torch.empty_like(lateral)
    _call("gf_upsample_add_ref", lateral.data_ptr(), src.data_ptr(), out.data_ptr(), b, h, w, src.shape[1], src.shape[2],
          c, _stream())
    return out


def add_posenc(x: torch.Tensor, pe: torch.Tensor) -> torch.Tensor:
    n, l, c = x.shape
    assert x.is_contiguous() and pe.is_contiguous() and pe.shape == (l, c)
    out = torch.empty_like(x)
    _call("gf_add_posenc", x.data_ptr(), pe.data_ptr(), out.data_ptr(), n, l, c, _stream())
    return out


def token_mask(mask: torch.Tensor, n: int, tokens: int) -> torch.Tensor:
    """data['mask0'] / data['mask1'] ([n, h_c, w_c] bool, 0 = padded; full_model.py:79-83) -> contiguous [n, tokens]
    uint8 on the device, the layout gf_mask_rows / gf_mask_fill_sim read."""
    if not mask.is_cuda:
        raise _lib.GeoFormerLibError("geoformer_b200 ops need CUDA tensors (no CPU fallback)")
    if mask.shape[0] != n or mask[0].numel() != tokens:
        raise ValueError(f"padding mask of shape {tuple(mask.shape)} does not cover {n} x {tokens} coarse tokens")
    m = mask.reshape(n, tokens)
    return (m if m.dtype == torch.bool else m != 0).contiguous().view(torch.uint8)


def mask_rows_(buf: torch.Tensor, mask: torch.Tensor, col0: int = 0, cols: Optional[int] = None) -> torch.Tensor:
    """In place buf[r, col0:col0+cols] *= mask[r] for a 0/1 row mask (linear_attention.py:37-43: Q * q_mask,
    K * kv_mask, values * kv_mask).  buf [rows, ld] fp32 or fp16, contiguous; mask uint8 [rows] (any shape, flattened)."""
    assert buf.dim() == 2 and buf.is_contiguous() and buf.dtype in (torch.float32, torch.float16)
    assert mask.dtype == torch.uint8 and mask.is_contiguous() and mask.numel() == buf.shape[0] and mask.device == buf.device
    rows, ld = buf.shape
    cols = ld - col0 if cols is None else cols
    _call("gf_mask_rows", buf.data_ptr(), buf.element_size(), rows, ld, col0, cols, mask.data_ptr(), _stream())
    return buf


def mask_fill_sim_(sim: torch.Tensor, mask0: torch.Tensor, mask1: torch.Tensor, fill: float = -1e9) -> torch.Tensor:
    """In place sim[b, i, j] = fill unless mask0[b, i] and mask1[b, j] (coarse_matching.py:120-124, INF = 1e9)."""
    _chk(sim)
    n, l, s = sim.shape
    assert sim.is_contiguous() and mask0.dtype == mask1.dtype == torch.uint8
    assert tuple(mask0.shape) == (n, l) and tuple(mask1.shape) == (n, s) and mask0.is_contiguous() and mask1.is_contiguous()
    _call("gf_mask_fill_sim", sim.data_ptr(), n, l, s, mask0.data_ptr(), mask1.data_ptr(), float(fill), _stream())
    return sim


def linattn(q: torch.Tensor, ldq: int, k: torch.Tensor, ldk: int, v: torch.Tensor, ldv: int, n: int, l: int, s: int,
            heads: int, dim: int) -> torch.Tensor:
    """Linear attention.  q/k/v are (views into) row-major buffers with row strides ldq/ldk/ldv (floats)."""
    dev = q.device
    nfl = _lib.load().gf_linattn_partial_floats(n, s, heads, dim)
    partial = torch.empty(nfl, device=dev, dtype=torch.float32)
    kv = torch.empty((n, heads, dim, dim), device=dev, dtype=torch.float32)
    ksum = torch.empty((n, heads, dim), device=dev, dtype=torch.float32)
    sfx = "_f16" if q.dtype == torch.float16 else ""          # fp16 storage of Q/K/V and of the message
    assert q.dtype == k.dtype == v.dtype
    _call("gf_linattn_reduce" + sfx, k.data_ptr(), ldk, v.data_ptr(), ldv, n, s, heads, dim, partial.data_ptr(),
              kv.data_ptr(), ksum.data_ptr(), _stream())
    out = torch.empty((n * l, heads * dim), device=dev, dtype=q.dtype)
    _call("gf_linattn_apply" + sfx, q.data_ptr(), ldq, kv.data_ptr(), ksum.data_ptr(), out.data_ptr(), n, l, s, heads,
              dim, _stream())
    return out


def linattn_window(q: torch.Tensor, ldq: int, k: torch.Tensor, ldk: int, v: torch.Tensor, ldv: int, n_windows: int,
                   tokens: int, heads: int, dim: int) -> torch.Tensor:
    assert q.dtype == k.dtype == v.dtype
    out = torch.empty((n_windows * tokens, heads * dim), device=q.device, dtype=q.dtype)
    _call("gf_linattn_window" + ("_f16" if q.dtype == torch.float16 else ""), q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, out.data_ptr(),
              n_windows, tokens, heads, dim, _stream())
    return out


def full_attention(q: torch.Tensor, ldq: int, k: torch.Tensor, ldk: int, v: torch.Tensor, ldv: int, n: int, l: int, s: int,
                   heads: int, dim: int) -> torch.Tensor:
    """LoFTR full attention (linear_attention.py:54-85): softmax(Q K^T / sqrt(dim)) V of every query row against all s key
    rows of its sample; q rows [n*l], k / v rows [n*s] (views with row strides ldq / ldk / ldv elements).  fp16 Q|K|V: the
    tcgen05 flash kernel (gf_dense_kv_h16 + gf_full_attention_tc, dim 32, heads*dim == 256); fp32: the FFMA kernel
    (accurate mode).  Returns the fp32 message [n*l, heads*dim]."""
    assert q.dtype == k.dtype == v.dtype
    dev = q.device
    out = torch.empty((n * l, heads * dim), device=dev, dtype=torch.float32)
    if q.dtype == torch.float16:
        s_pad = (s + 63) // 64 * 64
        kg = torch.empty((heads, n, s_pad, dim), device=dev, dtype=torch.float16)
        vt = torch.empty((heads, n, dim, s_pad), device=dev, dtype=torch.float16)
        cnt = torch.empty(n, device=dev, dtype=torch.int32)
        _call("gf_dense_kv_h16", k.data_ptr(), ldk, v.data_ptr(), ldv, n, s, heads, dim, s_pad, kg.data_ptr(), vt.data_ptr(),
              cnt.data_ptr(), _stream())
        _call("gf_full_attention_tc", q.data_ptr(), ldq, kg.data_ptr(), vt.data_ptr(), cnt.data_ptr(), out.data_ptr(), n, l,
              s, heads, dim, s_pad, _stream())
        return out
    _chk(q)
    _call("gf_full_attention", q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, out.data_ptr(), n, l, s, heads, dim,
          _stream())
    return out


def full_attention_window(q: torch.Tensor, ldq: int, k: torch.Tensor, ldk: int, v: torch.Tensor, ldv: int, n_windows: int,
                          tokens: int, heads: int, dim: int) -> torch.Tensor:
    """Full attention inside fine-level windows: window m's `tokens` query rows against window m's key / value rows.
    fp16 or fp32 Q|K|V; returns the fp32 message [n_windows*tokens, heads*dim]."""
    assert q.dtype == k.dtype == v.dtype
    out = torch.empty((n_windows * tokens, heads * dim), device=q.device, dtype=torch.float32)
    _call("gf_full_attention_window" + ("_f16" if q.dtype == torch.float16 else ""), q.data_ptr(), ldq, k.data_ptr(), ldk,
          v.data_ptr(), ldv, out.data_ptr(), n_windows, tokens, heads, dim, _stream())
    return out


def fine_layer_fused(x: torch.Tensor, src: torch.Tensor, wpack: torch.Tensor, n1w, n1b, n2w, n2b) -> torch.Tensor:
    """One fine-level LoFTR layer in a single kernel (csrc/fine_layer.cu).  x/src [m, 25, 128] fp32 contiguous."""
    _chk(x); _chk(src)
    m, t, c = x.shape
    assert (t, c) == (25, 128) and src.shape == x.shape and x.is_contiguous() and src.is_contiguous()
    assert wpack.dtype == torch.uint8 and wpack.shape == (30, 128, 128) and wpack.is_contiguous()
    y = torch.empty_like(x)
    _call("gf_fine_layer", x.data_ptr(), src.data_ptr(), wpack.data_ptr(), n1w.data_ptr(), n1b.data_ptr(), n2w.data_ptr(),
          n2b.data_ptr(), y.data_ptr(), m, _stream(), tag="[cross]" if src.data_ptr() != x.data_ptr() else "[self]")
    return y


# ------------------------------------------------------------------ coarse matching
def similarity(f0: torch.Tensor, f1: torch.Tensor, temperature: float, impl: Optional[str] = None) -> torch.Tensor:
    """sim[n,l,s] = (f0/sqrt(C)) . (f1/sqrt(C)) / temperature  (coarse_matching.py:110-119)."""
    _chk(f0); _chk(f1)
    n, l, c = f0.shape
    s = f1.shape[1]
    assert f0.is_contiguous() and f1.is_contiguous()
    sim = torch.empty((n, l, s), device=f0.device, dtype=torch.float32)
    in_scale = 1.0 / c ** 0.5
    if (impl or _SIM_IMPL) == "f16x3":
        a3 = torch.empty((n, l, 3 * c), device=f0.device, dtype=torch.float16)
        b3 = torch.empty((n, s, 3 * c), device=f0.device, dtype=torch.float16)
        _call("gf_pack_split_f16", f0.data_ptr(), a3.data_ptr(), n * l, c, in_scale, 0, _stream())
        _call("gf_pack_split_f16", f1.data_ptr(), b3.data_ptr(), n * s, c, in_scale, 1, _stream())
        _call("gf_similarity_f16x3", a3.data_ptr(), b3.data_ptr(), sim.data_ptr(), n, l, s, 3 * c,
              1.0 / temperature, _stream())
    else:
        _call("gf_similarity_ref", f0.data_ptr(), f1.data_ptr(), sim.data_ptr(), n, l, s, c, in_scale,
                  1.0 / temperature, _stream())
    return sim


def dual_softmax_(sim: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """In place sim -> conf = softmax(sim,1)*softmax(sim,2).  Returns (conf, conf_row_max, conf_col_max)."""
    n, l, s = sim.shape
    dev = sim.device
    rmax = torch.empty((n, l), device=dev); rsum = torch.empty((n, l), device=dev)
    cmax = torch.empty((n, s), device=dev); csum = torch.empty((n, s), device=dev)
    ws = torch.empty(_lib.load().gf_dual_softmax_workspace_floats(n, l, s), device=dev, dtype=torch.float32)
    _call("gf_dual_softmax_stats", sim.data_ptr(), n, l, s, rmax.data_ptr(), rsum.data_ptr(), cmax.data_ptr(),
              csum.data_ptr(), ws.data_ptr(), _stream())
    crmax = torch.empty((n, l), device=dev); ccmax = torch.empty((n, s), device=dev)
    _call("gf_dual_softmax_conf", sim.data_ptr(), n, l, s, rmax.data_ptr(), rsum.data_ptr(), cmax.data_ptr(),
              csum.data_ptr(), crmax.data_ptr(), ccmax.data_ptr(), _stream())
    return sim, crmax, ccmax


def conf_row_col_max(conf: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    n, l, s = conf.shape
    crmax = torch.empty((n, l), device=conf.device); ccmax = torch.empty((n, s), device=conf.device)
    _call("gf_conf_row_col_max", conf.data_ptr(), n, l, s, crmax.data_ptr(), ccmax.data_ptr(), _stream())
    return crmax, ccmax


def _compact(mj, mc, n, l, hw0c, hw1c, scale, dev):
    cap = n * l
    b_ids = torch.empty(cap, device=dev, dtype=torch.int64); i_ids = torch.empty_like(b_ids); j_ids = torch.empty_like(b_ids)
    mconf = torch.empty(cap, device=dev); k0 = torch.empty((cap, 2), device=dev); k1 = torch.empty((cap, 2), device=dev)
    counts = torch.empty(n + 1, device=dev, dtype=torch.int32)
    _call("gf_compact_coarse", mj.data_ptr(), mc.data_ptr(), n, l, hw0c[1], hw1c[1], float(scale), b_ids.data_ptr(),
          i_ids.data_ptr(), j_ids.data_ptr(), mconf.data_ptr(), k0.data_ptr(), k1.data_ptr(), counts.data_ptr(),
          counts.data_ptr() + 4 * n, cap, _stream())
    counts_h = counts.cpu()
    total = int(counts_h[n])
    return dict(b_ids=b_ids[:total], i_ids=i_ids[:total], j_ids=j_ids[:total], m_bids=b_ids[:total],
                mconf=mconf[:total], mkpts0_c=k0[:total], mkpts1_c=k1[:total]), counts_h[:n]


def coarse_match_fused(f0: torch.Tensor, f1: torch.Tensor, temperature: float, thr: float, border: int,
                       hw0c: Tuple[int, int], hw1c: Tuple[int, int], scale: float):
    """Whole coarse-matching stage without materialising the L x S matrix (two tcgen05 passes + vector MNN)."""
    _chk(f0); _chk(f1)
    n, l, c = f0.shape
    s = f1.shape[1]
    dev = f0.device
    a3 = torch.empty((n, l, 3 * c), device=dev, dtype=torch.float16)
    b3 = torch.empty((n, s, 3 * c), device=dev, dtype=torch.float16)
    in_scale = 1.0 / c ** 0.5
    _call("gf_pack_split_f16", f0.data_ptr(), a3.data_ptr(), n * l, c, in_scale, 0, _stream())
    _call("gf_pack_split_f16", f1.data_ptr(), b3.data_ptr(), n * s, c, in_scale, 1, _stream())
    ws = torch.empty(_lib.load().gf_coarse_match_fused_workspace_bytes(n, l, s), device=dev, dtype=torch.uint8)
    mj = torch.empty((n, l), device=dev, dtype=torch.int32)
    mc = torch.empty((n, l), device=dev, dtype=torch.float32)
    _call("gf_coarse_match_fused", a3.data_ptr(), b3.data_ptr(), n, l, s, 3 * c, 1.0 / temperature, float(thr), int(border),
          hw0c[0], hw0c[1], hw1c[0], hw1c[1], ws.data_ptr(), mj.data_ptr(), mc.data_ptr(), _stream())
    return _compact(mj, mc, n, l, hw0c, hw1c, scale, dev)


def mutual_nearest(conf: torch.Tensor, crmax: torch.Tensor, ccmax: torch.Tensor, thr: float, border: int,
                   hw0c: Tuple[int, int], hw1c: Tuple[int, int], scale: float):
    """MNN + threshold + border + ordered compaction.  Returns dict of exact-size tensors and per-sample counts.
    (One host sync to size the outputs, as the reference's torch.where does.)"""
    _chk(conf)
    n, l, s = conf.shape
    dev = conf.device
    mj = torch.empty((n, l), device=dev, dtype=torch.int32)
    mc = torch.empty((n, l), device=dev, dtype=torch.float32)
    _call("gf_mnn_select", conf.data_ptr(), n, l, s, float(thr), int(border), hw0c[0], hw0c[1], hw1c[0], hw1c[1],
              crmax.data_ptr(), ccmax.data_ptr(), mj.data_ptr(), mc.data_ptr(), _stream())
    cap = n * l
    b_ids = torch.empty(cap, device=dev, dtype=torch.int64); i_ids = torch.empty_like(b_ids); j_ids = torch.empty_like(b_ids)
    mconf = torch.empty(cap, device=dev); k0 = torch.empty((cap, 2), device=dev); k1 = torch.empty((cap, 2), device=dev)
    counts = torch.empty(n + 1, device=dev, dtype=torch.int32)
    _call("gf_compact_coarse", mj.data_ptr(), mc.data_ptr(), n, l, hw0c[1], hw1c[1], float(scale), b_ids.data_ptr(),
              i_ids.data_ptr(), j_ids.data_ptr(), mconf.data_ptr(), k0.data_ptr(), k1.data_ptr(), counts.data_ptr(),
              counts.data_ptr() + 4 * n, cap, _stream())
    counts_h = counts.cpu()
    total = int(counts_h[n])
    return dict(b_ids=b_ids[:total], i_ids=i_ids[:total], j_ids=j_ids[:total], m_bids=b_ids[:total],
                mconf=mconf[:total], mkpts0_c=k0[:total], mkpts1_c=k1[:total]), counts_h[:n]


# ------------------------------------------------------------------ geo attention
def geo_window_table(hmat: torch.Tensor, has_h: torch.Tensor, n: int, hw_src_c, hw_dst_px, w_dst_c: int, scale: int,
                     window: int) -> torch.Tensor:
    l = hw_src_c[0] * hw_src_c[1]
    widx = torch.empty((n, l, window * window), device=hmat.device, dtype=torch.int32)
    _call("gf_geo_window_table", hmat.data_ptr(), has_h.data_ptr(), n, hw_src_c[0], hw_src_c[1], hw_dst_px[0],
              hw_dst_px[1], w_dst_c, scale, window, widx.data_ptr(), _stream())
    return widx


def geo_self_attention(q, ldq, k, ldk, v, ldv, n, l, heads, dim, anchor_idx, anchor_cnt, max_cnt: int = 0,
                       impl: Optional[str] = None) -> torch.Tensor:
    """Full softmax attention of all l tokens against the anchor tokens of the same image.
    'tf32': per-head tcgen05 GEMMs over materialised score blocks; 'ref': fp32 flash-style FFMA kernel."""
    c = heads * dim
    out = torch.empty((n * l, c), device=q.device, dtype=torch.float32)
    mode = impl or _ATTN_IMPL
    if mode in ("tf32", "tf32_mat") and max_cnt > 0:
        s_pad = (max_cnt + 63) // 64 * 64
        dev = q.device
        if mode == "tf32":           # fused flash-style tcgen05 kernel (fp16 operands): scores never leave the SM
            kg = torch.empty((heads, n, s_pad, dim), device=dev, dtype=torch.float16)
            vt = torch.empty((heads, n, dim, s_pad), device=dev, dtype=torch.float16)
            if q.dtype == torch.float16:     # Q|K|V already fp16 (OUT16 projection): queries are read in place
                _call("gf_gather_anchor_kv_h16", k.data_ptr(), ldk, v.data_ptr(), ldv, n, l, heads, dim,
                      anchor_idx.data_ptr(), anchor_cnt.data_ptr(), anchor_idx.shape[1], s_pad, kg.data_ptr(),
                      vt.data_ptr(), _stream())
                q16, ld16 = q, ldq
            else:
                q16, ld16 = torch.empty((n * l, c), device=dev, dtype=torch.float16), c
                _call("gf_gather_anchor_kv_f16", q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, n, l, heads, dim,
                      anchor_idx.data_ptr(), anchor_cnt.data_ptr(), anchor_idx.shape[1], s_pad, q16.data_ptr(),
                      kg.data_ptr(), vt.data_ptr(), _stream())
            _call("gf_geo_self_attention_tc", q16.data_ptr(), ld16, kg.data_ptr(), vt.data_ptr(), out.data_ptr(), n, l,
                  heads, dim, s_pad, anchor_cnt.data_ptr(), _stream())
            return out
        kg = torch.empty((heads, n, s_pad, dim), device=dev, dtype=torch.float32)
        vt = torch.empty((heads, n, dim, s_pad), device=dev, dtype=torch.float32)
        _call("gf_gather_anchor_kv", k.data_ptr(), ldk, v.data_ptr(), ldv, n, l, heads, dim, anchor_idx.data_ptr(),
              anchor_cnt.data_ptr(), anchor_idx.shape[1], s_pad, kg.data_ptr(), vt.data_ptr(), _stream())
        sc = torch.empty((heads, n, l, s_pad), device=dev, dtype=torch.float32)
        for h in range(heads):
            _call("gf_gemm_tf32_batched", q.data_ptr() + 4 * h * dim, ldq, l * ldq, kg[h].data_ptr(), dim, s_pad * dim,
                  sc[h].data_ptr(), s_pad, l * s_pad, l, s_pad, dim, n, 1.0 / dim ** 0.5, _stream(), tag="[QK]")
        _call("gf_masked_softmax_rows", sc.data_ptr(), heads, n, l, s_pad, anchor_cnt.data_ptr(), _stream())
        for h in range(heads):
            _call("gf_gemm_tf32_batched", sc[h].data_ptr(), s_pad, l * s_pad, vt[h].data_ptr(), s_pad, dim * s_pad,
                  out.data_ptr() + 4 * h * dim, c, l * c, l, dim, s_pad, n, 1.0, _stream(), tag="[PV]")
        return out
    _call("gf_geo_self_attention", q.data_ptr(), ldq, k.data_ptr(), ldk, v.data_ptr(), ldv, out.data_ptr(), n, l,
              heads, dim, anchor_idx.data_ptr(), anchor_cnt.data_ptr(), anchor_idx.shape[1], _stream())
    return out


def geo_cross_attention(q, ldq, kp, ldk, vp, ldv, n, l, s, heads, dim, widx) -> torch.Tensor:
    out = torch.empty((n * l, heads * dim), device=q.device, dtype=q.dtype)
    _call("gf_geo_cross_attention" + ("_f16" if q.dtype == torch.float16 else ""), q.data_ptr(), ldq, kp.data_ptr(), ldk, vp.data_ptr(), ldv, out.data_ptr(), n,
              l, s, heads, dim, widx.data_ptr(), widx.shape[2], _stream())
    return out


def select_rows_(dst: torch.Tensor, src: torch.Tensor, flag: torch.Tensor, n: int, l: int, c: int) -> None:
    """dst[b] = src[b] for samples with flag[b] == 0 (per-sample skipped layers)."""
    _call("gf_select_rows", dst.data_ptr(), src.data_ptr(), flag.data_ptr(), n, l, c, _stream())


# ------------------------------------------------------------------ fine level
def fine_gather(fine_nhwc: torch.Tensor, b_ids, tok_ids, wc: int, stride: int, window: int,
                out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _, hf, wf, c = fine_nhwc.shape
    assert fine_nhwc.is_contiguous()
    m = b_ids.shape[0]
    if out is None:
        out = torch.empty((m, window * window, c), device=fine_nhwc.device, dtype=torch.float32)
    if out.dtype == torch.float16:
        assert fine_nhwc.dtype == torch.float16
        fn = "gf_fine_gather_f16_f16"
    else:
        fn = "gf_fine_gather_f16" if fine_nhwc.dtype == torch.float16 else "gf_fine_gather"
    _call(fn, fine_nhwc.data_ptr(), hf, wf, c, b_ids.data_ptr(), tok_ids.data_ptr(), m, wc, stride,
              window, out.data_ptr(), _stream())
    return out


def gather_rows(feat: torch.Tensor, b_ids, tok_ids, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _, l, c = feat.shape
    assert feat.is_contiguous()
    m = b_ids.shape[0]
    if out is None:
        out = torch.empty((m, c), device=feat.device, dtype=torch.float32)
    _call("gf_gather_rows", feat.data_ptr(), l, c, b_ids.data_ptr(), tok_ids.data_ptr(), m, out.data_ptr(), _stream())
    return out


def fine_match(f0: torch.Tensor, f1: torch.Tensor, temperature: float, thr: float, mkpts0_c, mkpts1_c, b_ids,
               window: int, coarse_scale: float, c2f: float, fine_scale: float, want_matrix: bool = False):
    m, ww, c = f0.shape
    dev = f0.device
    sel = torch.empty(m, device=dev, dtype=torch.int32); fi = torch.empty_like(sel); fj = torch.empty_like(sel)
    fconf = torch.empty(m, device=dev)
    fmat = torch.empty((m, ww, ww), device=dev) if want_matrix else None
    _call("gf_fine_match", f0.data_ptr(), f1.data_ptr(), m, ww, c, float(temperature), float(thr), sel.data_ptr(),
              fi.data_ptr(), fj.data_ptr(), fconf.data_ptr(), _ptr(fmat), _stream())
    k0 = torch.empty((m, 2), device=dev); k1 = torch.empty((m, 2), device=dev); mconf = torch.empty(m, device=dev)
    mb = torch.empty(m, device=dev, dtype=torch.int64); total = torch.empty(1, device=dev, dtype=torch.int32)
    _call("gf_compact_fine", sel.data_ptr(), fi.data_ptr(), fj.data_ptr(), fconf.data_ptr(), mkpts0_c.data_ptr(),
              mkpts1_c.data_ptr(), b_ids.data_ptr(), m, window, float(coarse_scale), float(c2f), float(fine_scale),
              k0.data_ptr(), k1.data_ptr(), mconf.data_ptr(), mb.data_ptr(), total.data_ptr(), _stream())
    t = int(total.item())
    return dict(mkpts0_f=k0[:t], mkpts1_f=k1[:t], mconf=mconf[:t], m_bids=mb[:t]), fmat, (sel, fi, fj, fconf)


# --------------------------------------------------------------------------------------------
# optional GPU RANSAC (csrc/ransac.cu) — replaces the host cv2.findHomography of geo_module.py:45-52
# --------------------------------------------------------------------------------------------
def ransac_homography(k0: torch.Tensor, k1: torch.Tensor, b_ids: torch.Tensor, counts: torch.Tensor, n: int,
                      hw0_c, hw1_c, scale: int, thr: float = 8.0, hyps: int = 1024, seed: int = 0):
    """k0/k1 [M,2] fp32 first-pass coarse matches, b_ids [M] int64, counts [n] int32 (device).
    Returns hm [2,n,9] (H and H^-1, fp32), has_h [n], inlier [M], aidx [2,n,cap], acnt [2,n]."""
    dev = k0.device
    _chk(k0); _chk(k1); _chk(b_ids, torch.int64); _chk(counts, torch.int32)
    assert k0.is_contiguous() and k1.is_contiguous()
    m = int(k0.shape[0])
    l0, l1 = hw0_c[0] * hw0_c[1], hw1_c[0] * hw1_c[1]
    cap = max(l0, l1)
    ws = torch.empty(_lib.load().gf_ransac_workspace_bytes(n, hyps), device=dev, dtype=torch.uint8)
    hm = torch.empty((2, n, 9), device=dev)
    has_h = torch.empty(n, device=dev, dtype=torch.int32)
    inlier = torch.empty(max(m, 1), device=dev, dtype=torch.int32)
    map0 = torch.empty((n, l0), device=dev, dtype=torch.int32); map1 = torch.empty((n, l1), device=dev, dtype=torch.int32)
    aidx = torch.zeros((2, n, cap), device=dev, dtype=torch.int32)
    acnt = torch.empty((2, n), device=dev, dtype=torch.int32)
    _call("gf_ransac_homography", k0.data_ptr(), k1.data_ptr(), b_ids.data_ptr(), counts.data_ptr(), m, n, hyps,
          float(thr), int(seed) & 0xffffffff, int(scale), l0, hw0_c[1], l1, hw1_c[1], ws.data_ptr(), hm[0].data_ptr(),
          hm[1].data_ptr(), has_h.data_ptr(), inlier.data_ptr(), map0.data_ptr(), map1.data_ptr(), aidx[0].data_ptr(),
          acnt[0].data_ptr(), aidx[1].data_ptr(), acnt[1].data_ptr(), cap, _stream(), tag="ransac")
    return hm, has_h, inlier[:m], aidx, acnt


# --------------------------------------------------------------------------------------------
# image ingest (csrc/ingest.cu) — the step before the path (eval_tool/immatch/utils/data_io.py:48-62)
# --------------------------------------------------------------------------------------------
def resize_gray_u8(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """cv2.resize(src, (wt, ht)) (INTER_LINEAR on uint8, bit-exact) followed by to_tensor's / 255:
    src uint8 [ho, wo] (device) -> dst fp32 [ht, wt] (device, contiguous; may be a slice of a batch tensor)."""
    if not src.is_cuda or not dst.is_cuda:
        raise _lib.GeoFormerLibError("geoformer_b200 ops need CUDA tensors (no CPU fallback)")
    assert src.dtype == torch.uint8 and src.dim() == 2 and src.is_contiguous()
    assert dst.dtype == torch.float32 and dst.dim() == 2 and dst.is_contiguous()
    _call("gf_resize_gray_u8", src.data_ptr(), src.shape[0], src.shape[1], dst.data_ptr(), dst.shape[0], dst.shape[1], _stream())
    return dst
