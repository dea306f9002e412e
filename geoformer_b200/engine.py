"""Host-side orchestration of the GeoFormer hot path on one B200.

Follows the stage order of the reference ``model/full_model.py:39-123``; every stage except the host RANSAC
(``cv2.findHomography``, geo_module.py:48, kept for parity by construction; ``model.ransac = "gpu"`` moves it to
csrc/ransac.cu) runs in hand-written sm_100a kernels reached through the C ABI (``geoformer_b200.ops``).  No cuDNN /
cuBLAS call exists in this package: the backbone is csrc/conv_tc.cu (fp16, product) or csrc/conv_ref.cu (fp32 FFMA,
accurate mode for the golden-match parity tests).
"""
from __future__ import annotations

import math
import os
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Tuple

import numpy as np
import torch

from . import ops
from .ops import EPI_ELU1, EPI_LN, EPI_RELU, EPI_TANH

_POOL: Optional[ThreadPoolExecutor] = None
# inference default: coarse matching without materialising the L x S matrix (conf_matrix is only produced when
# model.materialize is set); GF_FUSED_MATCHING=0 selects the materialised kernels
FUSED_MATCHING = os.environ.get("GF_FUSED_MATCHING", "1") != "0"
# fine-level LoFTR layers as one kernel per layer call (csrc/fine_layer.cu); GF_FUSED_FINE=0 selects the per-op kernels
FUSED_FINE_LAYER = os.environ.get("GF_FUSED_FINE", "1") != "0"


def _pool() -> ThreadPoolExecutor:
    global _POOL
    if _POOL is None:
        # GF_RANSAC_THREADS: host threads for the per-sample cv2.findHomography calls (default: one per core, <= 16)
        ranks = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))        # one process per GPU shares the host cores
        nthr = int(os.environ.get("GF_RANSAC_THREADS", "0")) or max(2, min(16, (os.cpu_count() or 2) // ranks))
        _POOL = ThreadPoolExecutor(max_workers=nthr)
        if os.environ.get("GF_CV2_THREADS"):            # OpenCV's own parallel_for_ width inside each findHomography call
            import cv2
            cv2.setNumThreads(int(os.environ["GF_CV2_THREADS"]))
    return _POOL


# --------------------------------------------------------------------------------------------
# weight packing
# --------------------------------------------------------------------------------------------
def _fold_bn(w: torch.Tensor, sd: Dict[str, torch.Tensor], bn: str, eps: float = 1e-5):
    """conv + eval-mode BN -> conv with bias: w' = w * g/sqrt(v+eps), b' = beta - mean * g/sqrt(v+eps)."""
    s = sd[bn + ".weight"].double() / torch.sqrt(sd[bn + ".running_var"].double() + eps)
    wf = (w.double() * s[:, None, None, None]).float()
    bf = (sd[bn + ".bias"].double() - sd[bn + ".running_mean"].double() * s).float()
    return wf, bf


def pack_conv3x3(w: torch.Tensor, b: Optional[torch.Tensor], cin_p: int, cout_p: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """[Cout,Cin,k,k] fp32 (+bias), k in {3, 1} -> tap-major K-major fp16 [cout_p, k*k, cin_k] and fp32 bias [cout_p]
    for gf_conv_f16 (cin_k = cin_p rounded up to a multiple of 64; all padding is zero)."""
    co, ci = w.shape[:2]
    taps = w.shape[2] * w.shape[3]
    cin_k = (cin_p + 63) // 64 * 64
    wt = torch.zeros((cout_p, taps, cin_k), dtype=torch.float32)
    wt[:co, :, :ci] = w.permute(0, 2, 3, 1).reshape(co, taps, ci)
    bias = torch.zeros(cout_p, dtype=torch.float32)
    if b is not None:
        bias[:co] = b
    return wt.to(device=device, dtype=torch.float16).contiguous(), bias.to(device)


def pack_fine_layer(wq, wk, wv, wm, w1, w2, device) -> torch.Tensor:
    """Weights of one fine-level layer as the 30 operand blocks [30][128 rows][128 B] gf_fine_layer streams per tile:
    12 fp32 blocks of Wq|Wk|Wv (n-chunk major, 32-float k-blocks), 8 fp32 blocks of mlp.0[:, :128], 2 fp16 blocks of
    merge (64-half k-blocks), 4 fp16 blocks of mlp.0[:, 128:], 4 fp16 blocks of mlp.2."""
    assert wq.shape == (128, 128) and w1.shape == (256, 256) and w2.shape == (128, 256)
    blocks = []

    def add(w, nchunks, k0, kblocks, half):
        kw = 64 if half else 32
        for nc in range(nchunks):
            for kb in range(kblocks):
                blk = w[nc * 128:(nc + 1) * 128, k0 + kb * kw:k0 + (kb + 1) * kw].detach().cpu()
                blk = blk.to(torch.float16 if half else torch.float32).contiguous()
                blocks.append(blk.view(torch.uint8).reshape(128, 128))

    add(torch.cat([wq, wk, wv], 0), 3, 0, 4, False)
    add(w1, 2, 0, 4, False)
    add(wm, 1, 0, 2, True)
    add(w1, 2, 128, 2, True)
    add(w2, 1, 0, 4, True)
    return torch.stack(blocks).contiguous().to(device)


class PackedWeights:
    """Device-resident, kernel-ready weights derived from a reference-schema state dict."""

    def __init__(self, sd: Dict[str, torch.Tensor], device: torch.device, backbone_dtype: torch.dtype):
        f32 = lambda t: t.detach().to(device=device, dtype=torch.float32).contiguous()
        f16 = lambda t: t.detach().to(device=device, dtype=torch.float16).contiguous()
        self.device = device
        self.backbone_dtype = backbone_dtype

        def enc(prefix: str, n_layers: int):
            layers = []
            for i in range(n_layers):
                p = f"{prefix}.layers.{i}."
                wq, wk, wv = sd[p + "q_proj.weight"], sd[p + "k_proj.weight"], sd[p + "v_proj.weight"]
                layers.append(dict(
                    wq=f32(wq), wkv=f32(torch.cat([wk, wv], 0)), wqkv=f32(torch.cat([wq, wk, wv], 0)),
                    wm=f32(sd[p + "merge.weight"]), w1=f32(sd[p + "mlp.0.weight"]), w2=f32(sd[p + "mlp.2.weight"]),
                    # fp16 copies for the GEMMs whose A operand is an fp16 intermediate (message, MLP hidden)
                    wm16=f16(sd[p + "merge.weight"]), w2_16=f16(sd[p + "mlp.2.weight"]),
                    n1w=f32(sd[p + "norm1.weight"]), n1b=f32(sd[p + "norm1.bias"]),
                    n2w=f32(sd[p + "norm2.weight"]), n2b=f32(sd[p + "norm2.bias"])))
            return layers

        def count(prefix: str) -> int:
            idx = {int(k[len(prefix) + 8:].split(".")[0]) for k in sd if k.startswith(prefix + ".layers.")}
            assert idx == set(range(len(idx))), f"{prefix}: non-contiguous layer indices {sorted(idx)}"
            return len(idx)

        # layer counts come from the state dict (== the config's layer_names; GeoFormer.__init__ builds the modules
        # from the config and forward() asserts the lengths agree), not from hard-coded 8 / 4 / 2
        self.coarse = enc("loftr_coarse", count("loftr_coarse"))
        self.geo = enc("geo_module.des_transformer", count("geo_module.des_transformer"))
        self.fine = enc("loftr_fine", count("loftr_fine"))
        for i, lw in enumerate(self.fine):
            p = f"loftr_fine.layers.{i}."
            if tuple(sd[p + "q_proj.weight"].shape) == (128, 128):
                lw["wpack"] = pack_fine_layer(sd[p + "q_proj.weight"], sd[p + "k_proj.weight"], sd[p + "v_proj.weight"],
                                              sd[p + "merge.weight"], sd[p + "mlp.0.weight"], sd[p + "mlp.2.weight"], device)
        wm = sd["fine_preprocess.merge_feat.weight"]
        cf = wm.shape[0]
        self.fp = dict(wd=f32(sd["fine_preprocess.down_proj.weight"]), bd=f32(sd["fine_preprocess.down_proj.bias"]),
                       wa=f32(wm[:, :cf]), wa16=f16(wm[:, :cf]), wb=f32(wm[:, cf:]),
                       bm=f32(sd["fine_preprocess.merge_feat.bias"]))

        # backbone: BN folded into weights + bias.  fp16 (product): tap-major K-major packs for the tcgen05 implicit GEMM
        # (csrc/conv_tc.cu); the 196-wide stage is zero-padded to 200 channels (16-byte rows for TMA): padded output
        # channels stay exactly 0 through ReLU / residual adds and padded input channels multiply zero weights.
        # fp32 (accurate mode): [taps][cin][cout] fp32 packs for the FFMA reference kernels (csrc/conv_ref.cu).
        cpad_to = 8
        bsd = {k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}

        def padc(c):
            return c if (c % cpad_to == 0 or c == 1) else (c + cpad_to - 1) // cpad_to * cpad_to

        def folded(name, bn=None):
            w = sd["backbone." + name + ".weight"]
            return _fold_bn(w, bsd, bn) if bn is not None else (w.float(), None)

        names = [("conv1", "bn1")]
        for li in (1, 2, 3):
            for bi in (0, 1):
                p = f"layer{li}.{bi}"
                names += [(p + ".conv1", p + ".bn1"), (p + ".conv2", p + ".bn2")]
                if li > 1 and bi == 0:
                    names.append((p + ".downsample.0", p + ".downsample.1"))
        names += [("layer3_outconv", None), ("layer2_outconv", None), ("layer1_outconv", None),
                  ("layer2_outconv2.0", "layer2_outconv2.1"), ("layer2_outconv2.3", None),
                  ("layer1_outconv2.0", "layer1_outconv2.1"), ("layer1_outconv2.3", None)]
        key = lambda name: name.replace(".downsample.0", ".down")
        self.bb_tc = self.bb_ref = None
        if backbone_dtype == torch.float16:
            t = {}
            for name, bn in names[1:]:
                w, b = folded(name, bn)
                t[key(name)] = pack_conv3x3(w, b, padc(w.shape[1]), padc(w.shape[0]), device)
            w7, b7 = folded("conv1", "bn1")                       # stem: [49 taps][128 channels]
            assert w7.shape == (128, 1, 7, 7)
            t["stem"] = (w7.reshape(128, 49).t().contiguous().to(device), b7.float().to(device))
            self.bb_tc = t
        elif backbone_dtype == torch.float32:
            r = {}
            for name, bn in names:
                w, b = folded(name, bn)
                co, ci, kh, kw = w.shape
                r[key(name)] = (w.permute(2, 3, 1, 0).reshape(kh * kw, ci, co).contiguous().to(device),
                                None if b is None else b.to(device))
            self.bb_ref = r
        else:
            raise ValueError(f"backbone dtype must be float16 (product) or float32 (accurate), got {backbone_dtype}")
        self._pe: Dict[Tuple[int, int, int], torch.Tensor] = {}
        self._pe_lock = threading.Lock()

    def pos_table(self, c: int, h: int, w: int) -> torch.Tensor:
        """[h*w, c] sinusoidal table in token-major layout.  Bug-compatible with the reference
        (position_encoding.py:28: ``-ln(1e4) / d_model // 2`` == -1.0, i.e. div_term[k] = exp(-2k))."""
        key = (c, h, w)
        t = self._pe.get(key)
        if t is not None:
            return t
        with self._pe_lock:                 # workers of MatchPipeline share this cache: build once, publish when complete
            if key in self._pe:
                return self._pe[key]
            ypos = torch.ones(h, w).cumsum(0).float().unsqueeze(0)
            xpos = torch.ones(h, w).cumsum(1).float().unsqueeze(0)
            div = torch.exp(torch.arange(0, c // 2, 2).float() * (-math.log(10000.0) / c // 2))[:, None, None]
            pe = torch.zeros(c, h, w)
            pe[0::4] = torch.sin(xpos * div); pe[1::4] = torch.cos(xpos * div)
            pe[2::4] = torch.sin(ypos * div); pe[3::4] = torch.cos(ypos * div)
            t = pe.permute(1, 2, 0).reshape(h * w, c).contiguous().to(self.device)      # pageable source: synchronous copy
            torch.cuda.current_stream(self.device).synchronize()
            self._pe[key] = t
        return t


# --------------------------------------------------------------------------------------------
# backbone (resnet_fpn.py:100-118)
# --------------------------------------------------------------------------------------------
def backbone_forward(pw: PackedWeights, img: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """[B,1,H,W] fp32 -> coarse NHWC [B,H/8,W/8,256] fp32, fine NHWC [B,H/2,W/2,128] (fp16 in product mode, fp32 in
    accurate mode); both contiguous."""
    return backbone_forward_tc(pw, img) if pw.bb_tc is not None else backbone_forward_ref(pw, img)


def backbone_forward_ref(pw: PackedWeights, img: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Accurate mode: the same network on the fp32 FFMA kernels of csrc/conv_ref.cu (NHWC fp32 throughout)."""
    r = pw.bb_ref

    def conv(name, t, act, residual=None, stride=1):
        wt, b = r[name]
        return ops.conv_ref(t, wt, b, residual, act, stride)

    def block(p, a):
        if (p + ".down") in r:
            y = conv(p + ".conv1", a, 1, stride=2)
            a = conv(p + ".down", a, 0, stride=2)
        else:
            y = conv(p + ".conv1", a, 1)
        return conv(p + ".conv2", y, 1, residual=a)

    b, _, h, w = img.shape
    x0 = conv("conv1", img.contiguous().view(b, h, w, 1), 1, stride=2)        # [B,1,H,W] == NHWC with one channel
    x1 = block("layer1.1", block("layer1.0", x0))
    x2 = block("layer2.1", block("layer2.0", x1))
    x3 = block("layer3.1", block("layer3.0", x2))
    x3o = conv("layer3_outconv", x3, 0)
    x2o = ops.upsample_add_ref(conv("layer2_outconv", x2, 0), x3o)
    x2o = conv("layer2_outconv2.3", conv("layer2_outconv2.0", x2o, 2), 0)
    x1o = ops.upsample_add_ref(conv("layer1_outconv", x1, 0), x2o)
    x1o = conv("layer1_outconv2.3", conv("layer1_outconv2.0", x1o, 2), 0)
    return x3o, x1o


def backbone_forward_tc(pw: PackedWeights, img: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Same network on this library's kernels only: every 3x3 and 1x1 convolution (stride 1 or 2) runs in the tcgen05
    implicit-GEMM kernel with BN, residual add and activation fused into its epilogue; the 7x7 stem is a register-
    tiled FFMA kernel and the FPN upsample+add one fused kernel.  Activations are NHWC fp16 throughout."""
    tc = pw.bb_tc

    def conv(name, t, act, residual=None, stride=1):
        wt, b = tc[name]
        return ops.conv(t, wt, b, residual, act, stride)

    def block(p, a):                                  # a: NHWC
        if (p + ".down") in tc:                       # stride-2 entry block: 3x3/s2 + ReLU, 1x1/s2 shortcut
            y = conv(p + ".conv1", a, 1, stride=2)
            a = conv(p + ".down", a, 0, stride=2)
        else:
            y = conv(p + ".conv1", a, 1)
        return conv(p + ".conv2", y, 1, residual=a)

    x0 = ops.stem_conv(img.contiguous(), *tc["stem"])
    x1 = block("layer1.1", block("layer1.0", x0))
    x2 = block("layer2.1", block("layer2.0", x1))
    x3 = block("layer3.1", block("layer3.0", x2))
    x3o = conv("layer3_outconv", x3, 0)
    x2o = ops.upsample_add(conv("layer2_outconv", x2, 0), x3o)
    x2o = conv("layer2_outconv2.3", conv("layer2_outconv2.0", x2o, 2), 0)
    x1o = ops.upsample_add(conv("layer1_outconv", x1, 0), x2o)
    x1o = conv("layer1_outconv2.3", conv("layer1_outconv2.0", x1o, 2), 0)
    return x3o.float().contiguous(), x1o          # the fine map stays fp16 NHWC: fine_gather reads it directly


# --------------------------------------------------------------------------------------------
# transformer layers
# --------------------------------------------------------------------------------------------
def _post_attention(lw: dict, x2d: torch.Tensor, msg: torch.Tensor, act: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """merge -> LN1 -> MLP(cat[x, msg]) -> LN2 -> residual   (transformer.py:53-60)."""
    h16 = ops.act16()
    m1 = ops.linear(msg, lw["wm16"] if msg.dtype == torch.float16 else lw["wm"], epi=EPI_LN, gamma=lw["n1w"], beta=lw["n1b"])
    h = ops.linear(x2d, lw["w1"], a2=m1, epi=act, out_f16=h16)
    return ops.linear(h, lw["w2_16"] if h16 else lw["w2"], epi=EPI_LN, gamma=lw["n2w"], beta=lw["n2b"], residual=x2d, out=out)


def _full_attention_layer(lw: dict, x: torch.Tensor, src: torch.Tensor, heads: int, out: Optional[torch.Tensor]):
    """LoFTR encoder layer with `attention: 'full'` (linear_attention.py:54-85): plain Q / K / V projections (no elu+1
    epilogue), softmax attention over all S source tokens, then the same merge / norm / MLP as the linear route.
    Product mode stores Q|K|V in fp16 for the tcgen05 flash kernel (heads x 32); otherwise fp32 for the FFMA kernel."""
    n, l, c = x.shape
    s = src.shape[1]
    d = c // heads
    x2d = x.reshape(n * l, c)
    a16 = ops.act16() and ops._ATTN_IMPL != "ref" and (c, d) == (256, 32)
    if x is src:
        qkv = ops.linear(x2d, lw["wqkv"], out_f16=a16)
        q, k, v, ldq, ldk = qkv, qkv[:, c:], qkv[:, 2 * c:], 3 * c, 3 * c
    else:
        q = ops.linear(x2d, lw["wq"], out_f16=a16)
        kv = ops.linear(src.reshape(n * s, c), lw["wkv"], out_f16=a16)
        k, v, ldq, ldk = kv, kv[:, c:], c, 2 * c
    msg = ops.full_attention(q, ldq, k, ldk, v, ldk, n, l, s, heads, d)
    return _post_attention(lw, x2d, msg, EPI_RELU, None if out is None else out.view(n * l, c)).view(n, l, c)


def loftr_layer(lw: dict, x: torch.Tensor, src: torch.Tensor, heads: int, out: Optional[torch.Tensor] = None,
                q_mask: Optional[torch.Tensor] = None, kv_mask: Optional[torch.Tensor] = None,
                attention: str = "linear") -> torch.Tensor:
    """LoFTR encoder layer with linear (default) or full softmax attention; x [n,L,C], src [n,S,C] -> [n,L,C] (written
    into `out` if given).  q_mask [n,L] / kv_mask [n,S] (uint8, 0 = padded token; optional; linear attention only): the
    feature-mapped Q / K rows and the value rows of padded tokens are cleared before the attention
    (linear_attention.py:37-43); the sequence length S that scales the values keeps counting them
    (linear_attention.py:45)."""
    if attention == "full":
        if q_mask is not None or kv_mask is not None:
            raise NotImplementedError("full attention with padding masks is not supported")
        return _full_attention_layer(lw, x, src, heads, out)
    assert attention == "linear", attention
    n, l, c = x.shape
    s = src.shape[1]
    d = c // heads
    x2d = x.reshape(n * l, c)
    a16 = ops.act16()
    if x is src:
        qkv = ops.linear(x2d, lw["wqkv"], epi=EPI_ELU1, act_cols=2 * c, out_f16=a16)          # [Q=elu+1 | K=elu+1 | V]
        if q_mask is not None and q_mask is kv_mask:
            ops.mask_rows_(qkv, q_mask)                                                       # one pass over Q | K | V
        else:
            if q_mask is not None:
                ops.mask_rows_(qkv, q_mask, 0, c)
            if kv_mask is not None:
                ops.mask_rows_(qkv, kv_mask, c, 2 * c)
        q, k, v, ldq, ldk = qkv, qkv[:, c:], qkv[:, 2 * c:], 3 * c, 3 * c
    else:
        q = ops.linear(x2d, lw["wq"], epi=EPI_ELU1, act_cols=c, out_f16=a16)
        kv = ops.linear(src.reshape(n * s, c), lw["wkv"], epi=EPI_ELU1, act_cols=c, out_f16=a16)
        if q_mask is not None:
            ops.mask_rows_(q, q_mask)
        if kv_mask is not None:
            ops.mask_rows_(kv, kv_mask)
        k, v, ldq, ldk = kv, kv[:, c:], c, 2 * c
    msg = ops.linattn(q, ldq, k, ldk, v, ldk, n, l, s, heads, d)
    return _post_attention(lw, x2d, msg, EPI_RELU, None if out is None else out.view(n * l, c)).view(n, l, c)


def coarse_transformer(pw: PackedWeights, x0: torch.Tensor, x1: torch.Tensor, names, heads: int,
                       mask0: Optional[torch.Tensor] = None, mask1: Optional[torch.Tensor] = None,
                       attention: str = "linear"):
    """loftr_module/transformer.py:82-104.  Same-size pairs run both images as one 2n-sample batch.
    attention: 'linear' or 'full' (the config's coarse.attention; every layer uses the same kind).
    mask0 [n,L] / mask1 [n,S] (uint8 token masks from ops.token_mask, both or neither): self layers mask queries and
    sources with the image's own mask, cross layers the queries with their own and the sources with the other image's
    (transformer.py:95-100)."""
    n = x0.shape[0]
    same = x0.shape == x1.shape
    assert (mask0 is None) == (mask1 is None), "padding masks come in pairs (full_model.py:82-83)"
    mm = None
    if same:
        X = torch.cat([x0, x1], 0)
        x0, x1 = X[:n], X[n:]
        if mask0 is not None:
            mm = torch.cat([mask0, mask1], 0)
    for lw, name in zip(pw.coarse, names):
        if name == "self":
            if same:
                X = loftr_layer(lw, X, X, heads, q_mask=mm, kv_mask=mm, attention=attention)
                x0, x1 = X[:n], X[n:]
            else:
                x0 = loftr_layer(lw, x0, x0, heads, q_mask=mask0, kv_mask=mask0, attention=attention)
                x1 = loftr_layer(lw, x1, x1, heads, q_mask=mask1, kv_mask=mask1, attention=attention)
        elif same:                                    # both results land in the halves of one fresh 2n-sample buffer
            Xn = torch.empty_like(X)
            y0 = loftr_layer(lw, x0, x1, heads, out=Xn[:n], q_mask=mask0, kv_mask=mask1, attention=attention)
            loftr_layer(lw, x1, y0, heads, out=Xn[n:], q_mask=mask1, kv_mask=mask0, attention=attention)   # sees the UPDATED feat0 (transformer.py:99-100)
            X = Xn
            x0, x1 = X[:n], X[n:]
        else:
            y0 = loftr_layer(lw, x0, x1, heads, q_mask=mask0, kv_mask=mask1, attention=attention)
            x0, x1 = y0, loftr_layer(lw, x1, y0, heads, q_mask=mask1, kv_mask=mask0, attention=attention)
    return x0, x1


def fine_layer(lw: dict, x: torch.Tensor, src: torch.Tensor, heads: int, attention: str = "linear") -> torch.Tensor:
    """LoFTR layer at the fine level: x/src [m, 25, 128]; one CTA per window for the linear attention, one warp per
    (window, head) for the full one (attention='full', which always takes the per-op path: the fused layer kernel is
    linear-only)."""
    m, t, c = x.shape
    d = c // heads
    if attention == "full":
        x2d = x.reshape(m * t, c)
        a16 = ops.act16() and ops._ATTN_IMPL != "ref" and d == 16
        if x is src:
            qkv = ops.linear(x2d, lw["wqkv"], out_f16=a16)
            q, k, v, ldq, ldk = qkv, qkv[:, c:], qkv[:, 2 * c:], 3 * c, 3 * c
        else:
            q = ops.linear(x2d, lw["wq"], out_f16=a16)
            kv = ops.linear(src.reshape(m * t, c), lw["wkv"], out_f16=a16)
            k, v, ldq, ldk = kv, kv[:, c:], c, 2 * c
        msg = ops.full_attention_window(q, ldq, k, ldk, v, ldk, m, t, heads, d)
        return _post_attention(lw, x2d, msg, EPI_RELU).view(m, t, c)
    assert attention == "linear", attention
    if FUSED_FINE_LAYER and ops.act16() and (t, c, heads) == (25, 128, 8) and "wpack" in lw:
        return ops.fine_layer_fused(x.contiguous(), src.contiguous(), lw["wpack"], lw["n1w"], lw["n1b"], lw["n2w"], lw["n2b"])
    x2d = x.reshape(m * t, c)
    a16 = ops.act16() and t == 25 and heads == 8 and d == 16
    if x is src:
        qkv = ops.linear(x2d, lw["wqkv"], epi=EPI_ELU1, act_cols=2 * c, out_f16=a16)
        q, k, v, ldq, ldk = qkv, qkv[:, c:], qkv[:, 2 * c:], 3 * c, 3 * c
    else:
        q = ops.linear(x2d, lw["wq"], epi=EPI_ELU1, act_cols=c, out_f16=a16)
        kv = ops.linear(src.reshape(m * t, c), lw["wkv"], epi=EPI_ELU1, act_cols=c, out_f16=a16)
        k, v, ldq, ldk = kv, kv[:, c:], c, 2 * c
    msg = ops.linattn_window(q, ldq, k, ldk, v, ldk, m, t, heads, d)
    return _post_attention(lw, x2d, msg, EPI_RELU).view(m, t, c)


# --------------------------------------------------------------------------------------------
# coarse matching
# --------------------------------------------------------------------------------------------
def coarse_matching(f0: torch.Tensor, f1: torch.Tensor, thr: float, temperature: float, border: int,
                    hw0_i, hw0_c, hw1_c, keep_conf: bool, mask0: Optional[torch.Tensor] = None,
                    mask1: Optional[torch.Tensor] = None):
    """utils/coarse_matching.py:90-212.  With padding masks (uint8 [n,L] / [n,S]) the logits of padded rows / columns are
    filled with -1e9 before the dual softmax (coarse_matching.py:120-124); that optional path runs on the materialising
    kernels (the fused matcher never holds the L x S matrix to fill).  `border` is 0 on this path (coarse_matching.py:30),
    which also makes mask_border_with_padding a no-op (coarse_matching.py:54-56)."""
    scale = hw0_i[0] / hw0_c[0]
    masked = mask0 is not None
    assert masked == (mask1 is not None), "padding masks come in pairs (coarse_matching.py:121)"
    assert not (masked and border > 0), "mask_border_with_padding (coarse_matching.py:54-68) is only built for border 0"
    if not keep_conf and not masked and ops._SIM_IMPL == "f16x3" and FUSED_MATCHING:
        matches, counts = ops.coarse_match_fused(f0, f1, temperature, thr, border, hw0_c, hw1_c, scale)
        return matches, counts, None
    sim = ops.similarity(f0, f1, temperature)
    if masked:
        ops.mask_fill_sim_(sim, mask0, mask1, -1e9)
    conf, crmax, ccmax = ops.dual_softmax_(sim)
    matches, counts = ops.mutual_nearest(conf, crmax, ccmax, thr, border, hw0_c, hw1_c, scale)
    return matches, counts, (conf if keep_conf else None)


# --------------------------------------------------------------------------------------------
# geo module
# --------------------------------------------------------------------------------------------
def _ransac_one(kp0: np.ndarray, kp1: np.ndarray, thr: float):
    import cv2
    if len(kp0) <= 8:                                    # geo_module.py:47
        return None, None
    M, mask = cv2.findHomography(kp0, kp1, cv2.RANSAC, thr)
    if M is None:
        return None, None
    return M, mask[:, 0] == 1


def geo_prepare_host(k0: np.ndarray, k1: np.ndarray, counts: np.ndarray, hw0_c, hw1_c, scale: int, ransac_thr: float):
    """Host side of geo_module.py:39-94: per-sample RANSAC, homographies (fp64 inverse, fp32 cast),
    anchor (inlier) token lists in ascending token order (== boolean-mask order).
    Only cv2.findHomography runs per sample (thread pool, GIL released); the bookkeeping around it is vectorised over
    the batch: one batched fp64 inverse, one boolean token map per image and one nonzero() for all samples."""
    n = len(counts)
    offs = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    k0i, k1i = k0.astype(np.int64), k1.astype(np.int64)
    kps = [(k0i[offs[b]:offs[b + 1]], k1i[offs[b]:offs[b + 1]]) for b in range(n)]
    if n > 1:
        res = list(_pool().map(lambda ab: _ransac_one(ab[0], ab[1], ransac_thr), kps))
    else:
        res = [_ransac_one(kps[0][0], kps[0][1], ransac_thr)]
    hm = np.zeros((2, n, 9), dtype=np.float32)
    has_h = np.array([1 if M is not None else 0 for M, _ in res], dtype=np.int32)
    if has_h.any():
        sel = np.flatnonzero(has_h)
        ms = np.stack([res[b][0] for b in sel])                                  # [k, 3, 3] fp64
        hm[0, sel] = ms.astype(np.float32).reshape(-1, 9)
        hm[1, sel] = torch.inverse(torch.from_numpy(ms)).to(torch.float32).numpy().reshape(-1, 9)
    # anchors: all first-pass matches of samples without a homography, the RANSAC inliers otherwise
    keep = np.ones(len(k0i), dtype=bool)
    for b in range(n):
        if has_h[b]:
            keep[offs[b]:offs[b + 1]] = res[b][1]
    bidx = np.repeat(np.arange(n, dtype=np.int64), counts)
    l0, l1 = hw0_c[0] * hw0_c[1], hw1_c[0] * hw1_c[1]
    lists = []
    for kk, wc, l in ((k0i, hw0_c[1], l0), (k1i, hw1_c[1], l1)):
        tok = (kk[:, 1] // scale) * wc + (kk[:, 0] // scale)
        m = np.zeros(n * l, dtype=bool)
        m[(bidx * l + tok)[keep]] = True
        flat = np.flatnonzero(m)                                                 # ascending (sample, token)
        cnt = np.bincount(flat // l, minlength=n).astype(np.int32)
        lists.append((flat % l, cnt))
    cap = max(1, int(max(lists[0][1].max(), lists[1][1].max())))
    aidx = np.zeros((2, n, cap), dtype=np.int32)
    acnt = np.zeros((2, n), dtype=np.int32)
    for side, (toks, cnt) in enumerate(lists):
        acnt[side] = cnt
        col = np.arange(len(toks)) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        aidx[side, np.repeat(np.arange(n), cnt), col] = toks
    return hm, has_h, aidx, acnt


def geo_self_layer(lw: dict, x: torch.Tensor, aidx: torch.Tensor, acnt: torch.Tensor, heads: int,
                   max_cnt: int = 0) -> torch.Tensor:
    """All tokens attend to the anchor tokens of their own image (geo_transformer/transformer.py:111-124)."""
    n, l, c = x.shape
    x2d = x.reshape(n * l, c)
    # product mode: Q|K|V stored fp16 (the flash kernel's operands are fp16 anyway: no conversion pass, half the gather)
    a16 = ops.act16() and ops._ATTN_IMPL == "tf32" and max_cnt > 0 and (heads, c // heads) == (4, 64)
    qkv = ops.linear(x2d, lw["wqkv"], out_f16=a16)
    att = ops.geo_self_attention(qkv, 3 * c, qkv[:, c:], 3 * c, qkv[:, 2 * c:], 3 * c, n, l, heads, c // heads, aidx, acnt,
                                 max_cnt)
    y = _post_attention(lw, x2d, att, EPI_TANH)
    ops.select_rows_(y, x2d, acnt, n, l, c)            # samples without anchors keep their features
    return y.view(n, l, c)


def geo_cross_layer(lw: dict, x0: torch.Tensor, x1: torch.Tensor, widx_in1: torch.Tensor, widx_in0: torch.Tensor,
                    has_h: torch.Tensor, heads: int):
    """Each token attends to its 25-token projected window in the other image; both directions read the
    PRE-layer features (geo_transformer/transformer.py:126-139)."""
    n, l, c = x0.shape
    s = x1.shape[1]
    d = c // heads
    a2d, b2d = x0.reshape(n * l, c), x1.reshape(n * s, c)
    a16 = ops.act16() and (heads, d) == (4, 64)         # Q|K|V and the message in fp16 storage (product mode)
    qkv0 = ops.linear(a2d, lw["wqkv"], out_f16=a16)
    qkv1 = ops.linear(b2d, lw["wqkv"], out_f16=a16)
    att0 = ops.geo_cross_attention(qkv0, 3 * c, qkv1[:, c:], 3 * c, qkv1[:, 2 * c:], 3 * c, n, l, s, heads, d, widx_in1)
    att1 = ops.geo_cross_attention(qkv1, 3 * c, qkv0[:, c:], 3 * c, qkv0[:, 2 * c:], 3 * c, n, s, l, heads, d, widx_in0)
    y0 = _post_attention(lw, a2d, att0, EPI_TANH)
    y1 = _post_attention(lw, b2d, att1, EPI_TANH)
    ops.select_rows_(y0, a2d, has_h, n, l, c)          # samples without a homography skip the layer
    ops.select_rows_(y1, b2d, has_h, n, s, c)
    return y0.view(n, l, c), y1.view(n, s, c)


def geo_module(pw: PackedWeights, x0: torch.Tensor, x1: torch.Tensor, first: dict, counts, hw0_i, hw1_i, hw0_c, hw1_c,
               names, heads: int, window: int, ransac_thr: float = 8.0, info: Optional[dict] = None,
               ransac: str = "cv2", ransac_hyps: int = 1024):
    n = x0.shape[0]
    dev = x0.device
    scale = int(hw0_i[0] // hw0_c[0])
    if ransac == "gpu":
        # optional device RANSAC (csrc/ransac.cu): no match coordinates leave the GPU; only 3n counters come back
        with ops.PROFILE.region("ransac_gpu"):
            cnt_d = torch.as_tensor(np.asarray(counts, dtype=np.int32)).to(dev, non_blocking=True)
            hm_d, has_h, _, aidx, acnt = ops.ransac_homography(first["mkpts0_c"], first["mkpts1_c"], first["b_ids"], cnt_d,
                                                               n, hw0_c, hw1_c, scale, ransac_thr, ransac_hyps)
            small = torch.cat([has_h[None], acnt]).cpu().numpy()
        has_h_np, acnt_np = small[0], small[1:]
        if info is not None:
            info.update(has_h=has_h_np.copy(), anchor_cnt=acnt_np.copy(), hmat=hm_d.cpu().numpy())
    elif ransac == "cv2":
        with ops.PROFILE.region("host:ransac"):
            k0 = first["mkpts0_c"].cpu().numpy()             # device -> host: RANSAC runs in OpenCV (geo_module.py:48)
            k1 = first["mkpts1_c"].cpu().numpy()
            hm, has_h_np, aidx_np, acnt_np = geo_prepare_host(k0, k1, np.asarray(counts), hw0_c, hw1_c, scale, ransac_thr)
        if info is not None:
            info.update(has_h=has_h_np.copy(), anchor_cnt=acnt_np.copy(), hmat=hm.copy())
        hm_d = torch.from_numpy(hm).to(dev, non_blocking=True)
        has_h = torch.from_numpy(has_h_np).to(dev, non_blocking=True)
        aidx = torch.from_numpy(aidx_np).to(dev, non_blocking=True)
        acnt = torch.from_numpy(acnt_np).to(dev, non_blocking=True)
    else:
        raise ValueError(f"ransac must be 'cv2' or 'gpu', got {ransac!r}")
    x0, x1 = x0.clone(), x1.clone()
    any_h = bool(has_h_np.any())
    if any_h:
        # tokens of image0 look into image1 through H; tokens of image1 look into image0 through H^-1
        widx_in1 = ops.geo_window_table(hm_d[0], has_h, n, hw0_c, hw1_i, hw1_c[1], scale, window)
        widx_in0 = ops.geo_window_table(hm_d[1], has_h, n, hw1_c, hw0_i, hw0_c[1], scale, window)
    for lw, name in zip(pw.geo, names):
        if name == "self":
            if acnt_np[0].any():
                x0 = geo_self_layer(lw, x0, aidx[0], acnt[0], heads, int(acnt_np[0].max()))
            if acnt_np[1].any():
                x1 = geo_self_layer(lw, x1, aidx[1], acnt[1], heads, int(acnt_np[1].max()))
        elif any_h:
            x0, x1 = geo_cross_layer(lw, x0, x1, widx_in1, widx_in0, has_h, heads)
    return x0, x1


# --------------------------------------------------------------------------------------------
# fine level
# --------------------------------------------------------------------------------------------
def fine_stage(pw: PackedWeights, fine0: torch.Tensor, fine1: torch.Tensor, g0: torch.Tensor, g1: torch.Tensor,
               m2: dict, hw0_i, hw0_c, hw1_c, hw0_f, window: int, heads: int, names, temperature: float, thr: float,
               want_matrix: bool, attention: str = "linear"):
    b_ids, i_ids, j_ids = m2["b_ids"], m2["i_ids"], m2["j_ids"]
    m = b_ids.shape[0]
    dev = fine0.device
    ww = window * window
    cf = fine0.shape[-1]
    stride = hw0_f[0] // hw0_c[0]
    # fine_preprocess.py:41-72.  merge_feat(cat[win, ctx]) = win Wa^T + (ctx Wb^T + b)
    w16 = ops.act16() and fine0.dtype == torch.float16 and cf % 64 == 0      # fp16 map -> fp16 windows -> fp16-operand merge
    win = torch.empty((2 * m, ww, cf), device=dev, dtype=torch.float16 if w16 else torch.float32)
    ops.fine_gather(fine0, b_ids, i_ids, hw0_c[1], stride, window, out=win[:m])
    ops.fine_gather(fine1, b_ids, j_ids, hw1_c[1], stride, window, out=win[m:])
    ctx = torch.empty((2 * m, g0.shape[-1]), device=dev)
    ops.gather_rows(g0, b_ids, i_ids, out=ctx[:m])
    ops.gather_rows(g1, b_ids, j_ids, out=ctx[m:])
    cw = ops.linear(ctx, pw.fp["wd"], bias=pw.fp["bd"])                          # down_proj            [2m, 128]
    cterm = ops.linear(cw, pw.fp["wb"], bias=pw.fp["bm"])                        # coarse half of merge [2m, 128]
    X = ops.linear(win.view(2 * m * ww, cf), pw.fp["wa16"] if w16 else pw.fp["wa"], rowbias=cterm,
                   rowbias_group=ww).view(2 * m, ww, cf)
    pre = X
    f0, f1 = X[:m], X[m:]
    for lw, name in zip(pw.fine, names):
        if name == "self":
            X = fine_layer(lw, X, X, heads, attention)
            f0, f1 = X[:m], X[m:]
        else:
            y0 = fine_layer(lw, f0, f1, heads, attention)
            y1 = fine_layer(lw, f1, y0, heads, attention)
            f0, f1 = y0, y1
    coarse_scale = hw0_i[0] / hw0_c[0]
    c2f = hw0_f[0] / hw0_c[0]
    fine_scale = hw0_i[0] / hw0_f[0]
    out, fmat, raw = ops.fine_match(f0.contiguous(), f1.contiguous(), temperature, thr, m2["mkpts0_c"], m2["mkpts1_c"],
                                    b_ids, window, coarse_scale, c2f, fine_scale, want_matrix)
    return out, fmat, dict(fine_in=pre, fine_out0=f0, fine_out1=f1, raw=raw)
