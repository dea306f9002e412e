"""Drop-in replacement for the reference ``model/full_model.py::GeoFormer``.

Same constructor, same ``forward(data) -> data`` contract over the ``data`` dict, same checkpoint
keys (253 tensors; ``matcher.`` prefixes stripped in ``load_state_dict``) and the same outputs
(``mkpts0_f`` / ``mkpts1_f`` / ``mconf`` / ``m_bids`` ...).  The modules below only *hold* parameters
under the reference's names; the arithmetic runs in libgeoformer_sm100.so (see ``geoformer_b200.engine``).
There is no CPU path: calling ``forward`` with CPU tensors raises.
"""
from __future__ import annotations

import os
import threading
from typing import Dict, Optional

import torch
import torch.nn as nn

from geoformer_b200 import engine, ops      # absolute: this file is also importable as top-level `model.full_model`
from .geo_config import default_cfg         # relative: the wrapper mutates the `default_cfg` of whichever name it imported


def _conv(cin, cout, k):
    return nn.Conv2d(cin, cout, kernel_size=k, bias=False)


class _Block(nn.Module):                      # parameter layout of resnet_fpn.py:15-31
    def __init__(self, cin, cout, stride):
        super().__init__()
        self.conv1, self.conv2 = _conv(cin, cout, 3), _conv(cout, cout, 3)
        self.bn1, self.bn2 = nn.BatchNorm2d(cout), nn.BatchNorm2d(cout)
        self.downsample = None if stride == 1 else nn.Sequential(_conv(cin, cout, 1), nn.BatchNorm2d(cout))


class _Backbone(nn.Module):                   # parameter layout of resnet_fpn.py:49-83
    def __init__(self, cfg):
        super().__init__()
        d0, (b1, b2, b3) = cfg["initial_dim"], cfg["block_dims"]
        self.conv1, self.bn1 = _conv(1, d0, 7), nn.BatchNorm2d(d0)
        self.layer1 = nn.Sequential(_Block(d0, b1, 1), _Block(b1, b1, 1))
        self.layer2 = nn.Sequential(_Block(b1, b2, 2), _Block(b2, b2, 1))
        self.layer3 = nn.Sequential(_Block(b2, b3, 2), _Block(b3, b3, 1))
        self.layer3_outconv = _conv(b3, b3, 1)
        self.layer2_outconv = _conv(b2, b3, 1)
        self.layer2_outconv2 = nn.Sequential(_conv(b3, b3, 3), nn.BatchNorm2d(b3), nn.LeakyReLU(), _conv(b3, b2, 3))
        self.layer1_outconv = _conv(b1, b2, 1)
        self.layer1_outconv2 = nn.Sequential(_conv(b2, b2, 3), nn.BatchNorm2d(b2), nn.LeakyReLU(), _conv(b2, b1, 3))
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")


class _EncoderLayer(nn.Module):               # parameter layout of loftr_module/transformer.py:10-35
    def __init__(self, d, act):
        super().__init__()
        self.q_proj, self.k_proj, self.v_proj, self.merge = (nn.Linear(d, d, bias=False) for _ in range(4))
        self.mlp = nn.Sequential(nn.Linear(2 * d, 2 * d, bias=False), act(), nn.Linear(2 * d, d, bias=False))
        self.norm1, self.norm2 = nn.LayerNorm(d), nn.LayerNorm(d)


class _Encoder(nn.Module):
    def __init__(self, d, n_layers, act=nn.ReLU, final_norm=False):
        super().__init__()
        self.layers = nn.ModuleList([_EncoderLayer(d, act) for _ in range(n_layers)])
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.xavier_uniform_(p)
        if final_norm:
            self.norm = nn.LayerNorm(d)       # present in checkpoints, unused in forward (geo_transformer/transformer.py:82)


class _FinePreprocess(nn.Module):             # fine_preprocess.py:9-28
    def __init__(self, dc, df):
        super().__init__()
        self.down_proj = nn.Linear(dc, df, bias=True)
        self.merge_feat = nn.Linear(2 * df, df, bias=True)
        for p in self.parameters():
            if p.dim() > 1:
                nn.init.kaiming_normal_(p, mode="fan_out", nonlinearity="relu")


class _GeoModule(nn.Module):
    def __init__(self, d, n_layers):
        super().__init__()
        self.des_transformer = _Encoder(d, n_layers, nn.Tanh, final_norm=True)


# "f16": tcgen05 implicit-GEMM backbone (product); "fp32": FFMA reference kernels (accurate mode for parity runs)
_BACKBONE_DTYPES = {"f16": torch.float16, "fp32": torch.float32}


def _attention_kinds(cfg) -> tuple:
    """(coarse, fine) attention of the LoFTR config: 'linear' (LinearAttention) or 'full' (FullAttention), read as
    loftr_module/transformer.py:22 does; anything else is refused."""
    kinds = tuple(cfg[level].get("attention", "linear") for level in ("coarse", "fine"))
    for level, kind in zip(("coarse", "fine"), kinds):
        if kind not in ("linear", "full"):
            raise ValueError(f"geoformer_b200.GeoFormer: {level}.attention must be 'linear' or 'full', got {kind!r}")
    return kinds


class GeoFormer(nn.Module):
    def __init__(self, loftr_config, geoformer_cfg=default_cfg):
        super().__init__()
        self.config = loftr_config
        self.geo_cfg = geoformer_cfg
        loftr_config["match_coarse"]["thr"] = geoformer_cfg["coarse_thr"]          # full_model.py:31
        dc, df = loftr_config["coarse"]["d_model"], loftr_config["fine"]["d_model"]
        self.backbone = _Backbone(loftr_config["resnetfpn"])
        self.loftr_coarse = _Encoder(dc, len(loftr_config["coarse"]["layer_names"]))
        self.fine_preprocess = _FinePreprocess(dc, df)
        self.loftr_fine = _Encoder(df, len(loftr_config["fine"]["layer_names"]))
        self.geo_module = _GeoModule(dc, len(geoformer_cfg["layer_names"]))
        # engine options (not part of the reference surface)
        self.backbone_precision = os.environ.get("GF_BACKBONE", "f16")
        # "cv2": host cv2.findHomography as the reference (geo_module.py:48); "gpu": csrc/ransac.cu (not bit-identical)
        self.ransac = os.environ.get("GF_RANSAC", "cv2")
        self.ransac_hyps = 1024
        # per-instance precision options, e.g. dict(linear="ref", similarity="ref", attention="ref", activations="f32") for
        # the accurate configuration; None = the module-level options of geoformer_b200.ops (ops.precision_scope)
        self.precision: Optional[dict] = None
        self.materialize = False       # also return conf_matrix / dect_conf_matrix / fine_matrix (training-side keys)
        self.capture = False           # keep per-stage tensors in data['_stages'] (tests)
        self._packed: Optional[engine.PackedWeights] = None
        self._tracked: list = []       # tensors the pack was built from (see _param_version)
        self._pack_lock = threading.Lock()
        if loftr_config["coarse"].get("temp_bug_fix", False):
            # position_encoding.py:26-28: only the (default) bug-compatible table is implemented
            raise NotImplementedError("geoformer_b200.GeoFormer: coarse.temp_bug_fix=True is not supported")
        _attention_kinds(loftr_config)
        if loftr_config["match_coarse"].get("match_type", "dual_softmax") != "dual_softmax":
            # sinkhorn (coarse_matching.py:100-108) needs a bin_score parameter that the checkpoint schema does not hold
            raise NotImplementedError("geoformer_b200.GeoFormer: match_coarse.match_type must be 'dual_softmax'")
        if not loftr_config.get("fine_concat_coarse_feat", True):
            # fine_preprocess.py:58-72: only the merge_feat route (coarse feature concatenated to the windows) is built
            raise NotImplementedError("geoformer_b200.GeoFormer: fine_concat_coarse_feat=False is not supported")

    # ---- parameter bookkeeping -----------------------------------------------------------------
    def load_state_dict(self, state_dict, *args, **kwargs):
        for k in list(state_dict.keys()):
            if k.startswith("matcher."):                                           # full_model.py:125-129
                state_dict[k.replace("matcher.", "", 1)] = state_dict.pop(k)
        self._packed = None
        return super().load_state_dict(state_dict, *args, **kwargs)

    def _apply(self, fn, *a, **kw):
        self._packed = None
        return super()._apply(fn, *a, **kw)

    def _param_version(self) -> int:
        """Sum of the in-place version counters of the parameters / buffers the current pack was built from: an in-place
        edit of any weight (optimizer step, `.copy_`, `.mul_` ...) changes it and the next forward repacks.  (Replacing a
        Parameter OBJECT is not seen here; load_state_dict / .to() reset the pack explicitly.)"""
        try:
            return sum(t._version for t in self._tracked)
        except RuntimeError:            # inference tensors do not track versions
            return 0

    def _weights(self, device) -> engine.PackedWeights:
        """Kernel-ready weights, packed once per device.  Thread-safe: MatchPipeline's workers call forward concurrently
        on their own streams, so packing happens under a lock and the packing stream is drained before the result is
        published (the H2D copies and casts are ordered on the packing stream only)."""
        pw = self._packed
        if pw is not None and pw.device == device and pw.version == self._param_version():
            return pw
        with self._pack_lock:
            ver = self._param_version()
            if self._packed is None or self._packed.device != device or self._packed.version != ver:
                if self.backbone_precision not in _BACKBONE_DTYPES:
                    raise ValueError(f"backbone_precision must be one of {sorted(_BACKBONE_DTYPES)}")
                ops.ensure_init(device)
                self._tracked = list(self.parameters()) + list(self.buffers())
                ver = self._param_version()
                pw = engine.PackedWeights({k: v for k, v in self.state_dict().items()}, device,
                                          _BACKBONE_DTYPES[self.backbone_precision])
                pw.version = ver
                cfg, gcfg = self.config, self.geo_cfg
                for got, names, what in ((pw.coarse, cfg["coarse"]["layer_names"], "coarse"),
                                         (pw.fine, cfg["fine"]["layer_names"], "fine"), (pw.geo, gcfg["layer_names"], "geo")):
                    assert len(got) == len(names), f"{what}: {len(got)} layers in the state dict, {len(names)} in the config"
                torch.cuda.current_stream(device).synchronize()
                self._packed = pw
            return self._packed

    # ---- forward ---------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, data: Dict[str, torch.Tensor]):
        img0, img1 = data["image0"], data["image1"]
        if (data.get("mask0") is None) != (data.get("mask1") is None):
            # full_model.py:82-83 reads both as soon as 'mask0' is present
            raise ValueError("geoformer_b200.GeoFormer: padding masks come in pairs (mask0 AND mask1)")
        for k in ("scale0", "scale1", "dataset_name"):
            # scale0/scale1 rescale mkpts*_c / the geo windows / mkpts*_f (coarse_matching.py:194, geo_module.py:39-42,
            # fine_matching2.py:96-115); dataset_name forces a match during training (coarse_matching.py:182).  Both
            # only exist in the training collations; ignoring them would silently change the result.
            if data.get(k) is not None:
                raise NotImplementedError(f"geoformer_b200.GeoFormer: data[{k!r}] is not supported (training-only key)")
        if data.get("mask0") is not None and _attention_kinds(self.config)[0] == "full":
            # FullAttention (linear_attention.py:75-77) fills masked logits with -inf: a fully padded query row is a softmax
            # over -inf only (NaN), which the next layer spreads into valid rows; there is no result to reproduce
            raise NotImplementedError("geoformer_b200.GeoFormer: coarse.attention='full' with padding masks is not supported")
        if not img0.is_cuda:
            raise RuntimeError("geoformer_b200.GeoFormer runs on CUDA (sm_100a) only; there is no CPU fallback")
        with torch.cuda.device(img0.device):       # kernels launch on the tensors' device and its current stream
            if self.precision:
                with ops.precision_scope(**self.precision):
                    return self._forward(data, img0, img1)
            return self._forward(data, img0, img1)

    def _forward(self, data, img0, img1):
        pw = self._weights(img0.device)
        cfg, gcfg = self.config, self.geo_cfg
        att_c, att_f = _attention_kinds(cfg)
        n = img0.shape[0]
        hw0_i, hw1_i = tuple(img0.shape[2:]), tuple(img1.shape[2:])
        data.update({"bs": torch.tensor(n), "hw0_i": torch.tensor(hw0_i), "hw1_i": torch.tensor(hw1_i)})
        stages = {} if self.capture else None

        R = ops.PROFILE.region
        # 1. CNN (resnet_fpn.py:100-118)
        with R("stage:backbone"):
            if hw0_i == hw1_i:
                c, f = engine.backbone_forward(pw, torch.cat([img0, img1], 0))
                c0, c1, f0, f1 = c[:n], c[n:], f[:n], f[n:]
            else:
                (c0, f0), (c1, f1) = engine.backbone_forward(pw, img0), engine.backbone_forward(pw, img1)
        hw0_c, hw1_c, hw0_f, hw1_f = tuple(c0.shape[1:3]), tuple(c1.shape[1:3]), tuple(f0.shape[1:3]), tuple(f1.shape[1:3])
        data.update({"hw0_c": torch.tensor(hw0_c), "hw1_c": torch.tensor(hw1_c),
                     "hw0_f": torch.tensor(hw0_f), "hw1_f": torch.tensor(hw1_f)})
        dc = c0.shape[-1]

        # 2. positional encoding + coarse transformer (full_model.py:69-84)
        # optional padding masks [N, h_c, w_c] (zero-padded batches; full_model.py:79-83): they reach the coarse
        # transformer and both coarse-matching calls, nothing else (geo module and fine level never see them)
        mk0 = mk1 = None
        if data.get("mask0") is not None:
            mk0 = ops.token_mask(data["mask0"], n, hw0_c[0] * hw0_c[1])
            mk1 = ops.token_mask(data["mask1"], n, hw1_c[0] * hw1_c[1])
        with R("stage:coarse_transformer"):
            x0 = ops.add_posenc(c0.reshape(n, -1, dc), pw.pos_table(dc, *hw0_c))
            x1 = ops.add_posenc(c1.reshape(n, -1, dc), pw.pos_table(dc, *hw1_c))
            t0, t1 = engine.coarse_transformer(pw, x0, x1, cfg["coarse"]["layer_names"], cfg["coarse"]["nhead"], mk0, mk1,
                                               attention=att_c)

        # 3. coarse matching -> geo module -> coarse matching (full_model.py:87-90)
        thr = cfg["match_coarse"]["thr"]
        temp = cfg["match_coarse"]["dsmax_temperature"]
        with R("stage:coarse_matching_1"):
            m1, counts1, conf1 = engine.coarse_matching(t0.contiguous(), t1.contiguous(), thr, temp, 0, hw0_i, hw0_c,
                                                        hw1_c, self.materialize, mk0, mk1)
        ginfo = {} if self.capture else None
        with R("stage:geo_module(+host RANSAC)"):
            g0, g1 = engine.geo_module(pw, x0, x1, m1, counts1, hw0_i, hw1_i, hw0_c, hw1_c, gcfg["layer_names"],
                                       gcfg["nhead"], gcfg["window_size"], info=ginfo, ransac=self.ransac,
                                       ransac_hyps=self.ransac_hyps)
        with R("stage:coarse_matching_2"):
            m2, counts2, conf2 = engine.coarse_matching(g0, g1, thr, temp, 0, hw0_i, hw0_c, hw1_c, self.materialize,
                                                        mk0, mk1)
        data.update(m2)
        if self.materialize:
            data.update({"dect_conf_matrix": conf1, "conf_matrix": conf2})

        # 4/5. fine level (fine_preprocess.py, loftr_fine, fine_matching2.py)
        w = cfg["fine_window_size"]
        data.update({"W": torch.tensor(w)})
        if m2["b_ids"].shape[0] == 0:
            data.update({"mkpts0_f": m2["mkpts0_c"], "mkpts1_f": m2["mkpts1_c"],
                         "fine_matrix": torch.empty(0, w * w, w * w, device=img0.device)})
            fstages = {}
        else:
            with R("stage:fine"):
                out, fmat, fstages = engine.fine_stage(pw, f0, f1, g0, g1, m2, hw0_i, hw0_c, hw1_c, hw0_f, w,
                                                       cfg["fine"]["nhead"], cfg["fine"]["layer_names"],
                                                       gcfg["fine_temperature"], gcfg["fine_thr"], self.materialize,
                                                       attention=att_f)
            data.update(out)
            if self.materialize:
                data["fine_matrix"] = fmat
        if stages is not None:
            stages.update(cnn_c0=c0, cnn_c1=c1, fine0=f0, fine1=f1, pe0=x0, pe1=x1, coarse0=t0, coarse1=t1,
                          first=m1, counts_first=counts1, geo0=g0, geo1=g1, geo_info=ginfo, counts=counts2, **fstages)
            data["_stages"] = stages
        return data
