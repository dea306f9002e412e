"""CPU checker for LoFTR's full softmax attention (`attention: 'full'` in the coarse / fine config).

TEST INFRASTRUCTURE ONLY, like `oracle/geoformer_oracle.py` (whose building blocks it reuses unchanged): an fp32
restatement of FullAttention (model/loftr_src/loftr/loftr_module/linear_attention.py:54-85), of the LoFTR encoder layer
that uses it (loftr_module/transformer.py:22, 37-60) and of the forward (model/full_model.py:39-123) with the attention
kind chosen per level.  The reference cannot be run for this option, so no reference-generated golden exists: these lines
are the checker; everything around the attention is the oracle's and pinned by the linear-route goldens.  Padding masks
are not restated (the product refuses them with full attention: a fully masked row is NaN in the reference)."""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from oracle import geoformer_oracle as O


def full_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """linear_attention.py:54-85 without masks (dropout is off at inference): q [N,L,H,D], k / v [N,S,H,D], the plain
    projections (no elu+1 map) -> [N,L,H,D]."""
    QK = torch.einsum("nlhd,nshd->nlsh", q, k)
    softmax_temp = 1.0 / q.size(3) ** 0.5
    A = torch.softmax(softmax_temp * QK, dim=2)
    return torch.einsum("nlsh,nshd->nlhd", A, v).contiguous()


def encoder_layer(P: Dict[str, torch.Tensor], pre: str, x: torch.Tensor, src: torch.Tensor, nhead: int) -> torch.Tensor:
    """LoFTREncoderLayer with attention='full' (transformer.py:37-60)."""
    n, _, c = x.shape
    d = c // nhead
    q = F.linear(x, P[pre + ".q_proj.weight"]).view(n, -1, nhead, d)
    k = F.linear(src, P[pre + ".k_proj.weight"]).view(n, -1, nhead, d)
    v = F.linear(src, P[pre + ".v_proj.weight"]).view(n, -1, nhead, d)
    m = F.linear(full_attention(q, k, v).view(n, -1, c), P[pre + ".merge.weight"])
    m = F.layer_norm(m, (c,), P[pre + ".norm1.weight"], P[pre + ".norm1.bias"], 1e-5)
    m = F.relu(F.linear(torch.cat([x, m], dim=2), P[pre + ".mlp.0.weight"]))
    m = F.layer_norm(F.linear(m, P[pre + ".mlp.2.weight"]), (c,), P[pre + ".norm2.weight"], P[pre + ".norm2.bias"], 1e-5)
    return x + m


def local_feature_transformer(P, pre: str, f0: torch.Tensor, f1: torch.Tensor, layer_names, nhead: int,
                              attention: str) -> Tuple[torch.Tensor, torch.Tensor]:
    """transformer.py:82-104 with one attention kind for every layer; the cross update of f1 sees the updated f0."""
    if attention == "linear":
        return O.local_feature_transformer(P, pre, f0, f1, layer_names, nhead)
    assert attention == "full", attention
    for i, name in enumerate(layer_names):
        lp = f"{pre}.layers.{i}"
        if name == "self":
            f0, f1 = encoder_layer(P, lp, f0, f0, nhead), encoder_layer(P, lp, f1, f1, nhead)
        else:
            f0 = encoder_layer(P, lp, f0, f1, nhead)
            f1 = encoder_layer(P, lp, f1, f0, nhead)
    return f0, f1


def forward(P, image0: torch.Tensor, image1: torch.Tensor, cfg: Optional[dict] = None,
            coarse: str = "full", fine: str = "full") -> Dict[str, torch.Tensor]:
    """full_model.py:39-123 (the steps of O.forward, no masks) with coarse.attention / fine.attention = coarse / fine."""
    cfg = {**O.DEFAULT_CFG, **(cfg or {})}
    n = image0.shape[0]
    hw0_i, hw1_i = tuple(image0.shape[2:]), tuple(image1.shape[2:])
    if hw0_i == hw1_i:
        fc, ff = O.backbone(P, torch.cat([image0, image1], 0))
        (c0, c1), (ff0, ff1) = fc.split(n), ff.split(n)
    else:
        (c0, ff0), (c1, ff1) = O.backbone(P, image0), O.backbone(P, image1)
    hw0_c, hw1_c = tuple(c0.shape[2:]), tuple(c1.shape[2:])
    hw0_f = tuple(ff0.shape[2:])
    x0, x1 = O.add_pe_flatten(c0), O.add_pe_flatten(c1)
    t0, t1 = local_feature_transformer(P, "loftr_coarse", x0, x1, cfg["coarse_layers"], cfg["coarse_nhead"], coarse)
    m1 = O.coarse_match(O.dual_softmax_conf(t0, t1, cfg["coarse_temperature"]), cfg["coarse_thr"], hw0_i, hw0_c, hw1_c,
                        cfg["border_rm"])
    geo = O.geo_prepare(m1, n, hw0_i, hw1_i, hw0_c, hw1_c, cfg)
    g0, g1 = O.geo_transformer(P, x0, x1, geo, hw0_c, hw1_c, cfg)
    m2 = O.coarse_match(O.dual_softmax_conf(g0, g1, cfg["coarse_temperature"]), cfg["coarse_thr"], hw0_i, hw0_c, hw1_c,
                        cfg["border_rm"])
    stride = hw0_f[0] // hw0_c[0]
    w0, w1 = O.fine_preprocess(P, ff0, ff1, g0, g1, m2["b_ids"], m2["i_ids"], m2["j_ids"], cfg["fine_window"], stride)
    out = dict(m2, coarse0=t0, coarse1=t1)
    if w0.shape[0] == 0:
        out.update(mkpts0_f=m2["mkpts0_c"], mkpts1_f=m2["mkpts1_c"])
        return out
    w0, w1 = local_feature_transformer(P, "loftr_fine", w0, w1, cfg["fine_layers"], cfg["fine_nhead"], fine)
    fconf = O.dual_softmax_conf(w0, w1, cfg["fine_temperature"])
    out.update(O.fine_match(fconf, cfg["fine_thr"], m2["mkpts0_c"], m2["mkpts1_c"], m2["b_ids"], hw0_i, hw0_c, hw0_f,
                            cfg["fine_window"]))
    return out
