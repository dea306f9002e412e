"""GPU tests of LoFTR's full softmax attention (`attention: 'full'` in the coarse / fine config,
loftr_module/linear_attention.py:54-85), from the kernels up to GeoFormer.forward:

  A  the coarse tcgen05 flash kernel at head dim 32 (geo_flash_attn_kernel<32>, dense keys) at the shipped shape: self
     attention over 32 x 4800 tokens (16 pairs at 480x640) and cross attention 4800 <-> 3000 (partial last key tile),
     with logits shaped so that the lazy reference maximum is raised; and the fp32 FFMA kernel on the same inputs;
  B  the fine-level window kernel (one warp per (window, head), 25 tokens, 8 x 16), fp16 and fp32 storage;
  C  one LoFTR layer with attention='full' against the checker's encoder_layer (tests/loftr_full_oracle.py), coarse and
     fine, self and cross;
  D  the whole forward with both levels 'full': accurate mode reproduces the checker's forward integer outputs exactly, the
     shipped configuration keeps the coarse-transformer features close at 480x640.

Kernel references are fp64 on the CPU on the same fp16-rounded operands the kernel reads (large ones on a fixed subset
of rows).  A test that exists to reach a branch asserts on the host that its inputs reach it."""
import copy
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from geoformer_b200 import synth
from oracle import geoformer_oracle as O
from tests import loftr_full_oracle as LF
from tests.util import load_golden, stage_case_inputs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from geoformer_b200 import ops as _ops
    assert torch.cuda.is_available(), "GPU tests need a B200"
    _ops.ensure_init(torch.device("cuda:0"))
    return _ops


def dev(t):
    return t.cuda().contiguous()


ACCURATE = dict(linear="ref", similarity="ref", attention="ref", activations="f32")
SHIPPED = dict(linear="tf32", similarity="f16x3", attention="tf32", activations="f16")


# ------------------------------------------------------------------------------------------- A: coarse kernel, d = 32
HEADS, DIM = 8, 32
KBK, KRING, KLAZY = 64, 4, 8.0               # flash_attn.cu: keys per tile, K / V^T ring stages, lazy window (log2 units)
LOG2E = 1.4426950408889634
# (n, l, s, checked samples): self at the shipped batch, cross both ways between 4800 and 3000 tokens
COARSE_CASES = {"self": (32, 4800, 4800, (0, 13, 31)), "cross_4800_3000": (4, 4800, 3000, (0, 3)),
                "cross_3000_4800": (4, 3000, 4800, (1, 2))}


def _coarse_inputs(n, l, s, seed):
    """fp16 Q [n, l, h, d], K / V [n, s, h, d] with logits shaped per head.  Each head has a unit direction u; Q and K are
    random orthogonal to u, queries get +sqrt(d) u on even rows and -sqrt(d) u on odd rows, the key j gets r_h(j) u, so
    logit = q.k / sqrt(d) = noise +- r_h(j):
      head 0: r = 1.6 per key tile: the '+' rows' maximum climbs and is raised every ~4 tiles (logits up to ~120);
      head 1: r climbs 4.9 logits (7.1 log2 units) over the whole sequence: P approaches 2^8 without a raise;
      head 3: the last key spikes 40 logits: a raise by ~58 log2 units in the last tile;
      heads 2, 4..7: plain random logits."""
    h, d = HEADS, DIM
    g = torch.Generator().manual_seed(seed)
    u = torch.randn(h, d, generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    perp = lambda x: x - (x * u).sum(-1, keepdim=True) * u
    q = perp(torch.randn(n, l, h, d, generator=g))
    k = perp(torch.randn(n, s, h, d, generator=g))
    v = torch.randn(n, s, h, d, generator=g)
    sign = 1.0 - 2.0 * (torch.arange(l) % 2).float()
    q = q + math.sqrt(d) * sign[None, :, None, None] * u
    tile = (torch.arange(s) // KBK).float()
    tiles = (s + KBK - 1) // KBK
    ramp = torch.zeros(s, h)
    ramp[:, 0] = 1.6 * tile
    ramp[:, 1] = 4.9 * tile / max(tiles - 1, 1)
    ramp[s - 1, 3] = 40.0
    k = k + ramp[None, :, :, None] * u
    return q.half(), k.half(), v.half()


def _rows(l):
    """Checked query rows: the first 128-row tile, the partial last tile and 300 seeded random rows in between."""
    g = torch.Generator().manual_seed(21)
    last = (l - 1) // 128 * 128
    return torch.unique(torch.cat([torch.arange(128), torch.randint(128, last, (300,), generator=g), torch.arange(last, l)]))


def _reference(q, k, v, rows):
    """fp64 attention of the checked rows of one sample (q [l, h, d], k / v [s, h, d] fp64) plus a replay of the kernel's
    lazy-maximum rule (tile maxima in log2 units against a reference maximum raised only on a lead > KLAZY), and two
    deliberately broken results: the recurrence without any rescale, and softmax without the 1/sqrt(d) scale."""
    d = q.shape[-1]
    s_ = torch.einsum("rhd,jhd->rhj", q[rows], k) / math.sqrt(d)
    want = torch.einsum("rhj,jhd->rhd", torch.softmax(s_, -1), v)
    no_scale = torch.einsum("rhj,jhd->rhd", torch.softmax(s_ * math.sqrt(d), -1), v)
    cnt = k.shape[0]
    tiles = (cnt + KBK - 1) // KBK
    s2 = F.pad(s_ * LOG2E, (0, tiles * KBK - cnt), value=-math.inf).view(len(rows), HEADS, tiles, KBK)
    del s_
    tm2 = s2.amax(-1)                                                               # [R, h, T]
    m2, raised, lead = torch.empty_like(tm2), torch.zeros_like(tm2, dtype=torch.bool), torch.full_like(tm2, -math.inf)
    m = m2[..., 0] = tm2[..., 0]
    for t in range(1, tiles):
        lead[..., t] = tm2[..., t] - m
        raised[..., t] = lead[..., t] > KLAZY
        m = torch.where(raised[..., t], tm2[..., t], m)
        m2[..., t] = m
    p = torch.exp2(s2 - m2[..., None])                                              # the kernel's P of every tile
    del s2
    vt = F.pad(v, (0, 0, 0, 0, 0, tiles * KBK - cnt)).view(tiles, KBK, HEADS, d)
    o_t = torch.einsum("rhtj,tjhd->rhtd", p, vt)
    l_t = p.sum(-1)
    w = torch.exp2(m2 - m2[..., -1:])                                               # rescale factors up to the last tile
    exact = (o_t * w[..., None]).sum(2) / (l_t * w).sum(2)[..., None]
    assert (exact - want).abs().max().item() <= 1e-9                                # the replay is the same softmax
    return dict(want=want, vmin=v.amin(0), vmax=v.amax(0), vabs=v.abs().max().item(), tiles=tiles, raised=raised,
                lead=lead, p_last=p[..., -1, :].amax(-1), no_rescale=o_t.sum(2) / l_t.sum(2)[..., None], no_scale=no_scale)


@pytest.fixture(scope="module")
def coarse_cases():
    out = {}
    for name, (n, l, s, checked) in COARSE_CASES.items():
        q, k, v = _coarse_inputs(n, l, s, seed=30 + len(out))
        rows = _rows(l)
        refs = {b: _reference(q[b].double(), k[b].double(), v[b].double(), rows) for b in checked}
        out[name] = dict(q=q, k=k, v=v, rows=rows, refs=refs, shape=(n, l, s))
    return out


def _tol(r):
    """Per element: O and l come from the same fp16-rounded P (2^-11 relative each), so the error of O / l is bounded by
    2^-11 * max_i |v_i - out| on top of fp32 round-off: bar 2^-10 * max_i |v_i - want| + 1e-5."""
    spread = torch.maximum(r["vmax"] - r["want"], r["want"] - r["vmin"])
    return 2.0 ** -10 * spread + 1e-5


def test_coarse_cases_reach_the_lazy_rescale_and_catch_broken_kernels(coarse_cases):
    """Premise of the shipped-shape cases (host only): the '+' rows of head 0 are raised many times, head-1 rows lead by
    (6, 8] log2 units without a raise, the last-tile spike of head 3 raises, warps mix raised and unraised lanes, the K /
    V ring wraps, the cross cases end on a partial key tile; and a kernel that skipped the rescale or dropped the
    1/sqrt(32) scale would miss the bar of _tol by more than 10x."""
    case = coarse_cases["self"]
    rows, r0 = case["rows"], case["refs"][0]
    plus = rows % 2 == 0
    assert r0["tiles"] > 2 * KRING
    n_raise = r0["raised"].sum(-1)                                                  # [R, h]
    assert n_raise[plus, 0].min().item() >= 10, n_raise[plus, 0].min()
    assert n_raise[~plus, 0].max().item() == 0
    lead_kept = torch.where(r0["raised"], torch.full_like(r0["lead"], -math.inf), r0["lead"]).amax(-1)
    near = (lead_kept[:, 1] > 6) & (lead_kept[:, 1] <= KLAZY)
    assert near.sum().item() >= 20, near.sum()
    assert r0["raised"][plus, 3, -1].all()
    assert (r0["p_last"][~plus, 0] < 2.0 ** -25).all()                              # '-' rows of head 0 underflow fp16
    first = r0["raised"][:128].view(4, 32, HEADS, -1)
    mixed = first.any(1) & ~first.all(1)
    assert mixed[:, 0].any(-1).all(), "every warp has raised and unraised lanes in the same tile"
    for name in ("cross_4800_3000",):
        assert coarse_cases[name]["shape"][2] % KBK != 0                            # partial last key tile
    for name, c in coarse_cases.items():
        for b, r in c["refs"].items():
            tol = _tol(r)
            for broken in ("no_rescale", "no_scale"):
                ratio = ((r[broken] - r["want"]).abs() / tol).max().item()
                assert ratio > 10, (name, b, broken, ratio)


@pytest.mark.parametrize("route", ["f16", "accurate"])
@pytest.mark.parametrize("case", list(COARSE_CASES))
def test_coarse_full_attention_shipped_shape(ops, coarse_cases, case, route):
    """ops.full_attention on the engine's layouts: 'f16' (product: fp16 Q|K|V read in place, gf_dense_kv_h16 +
    gf_full_attention_tc) and 'accurate' (fp32 Q|K|V holding the same values, gf_full_attention, fp32 FFMA).  Self reads
    one [n*l, 768] Q|K|V buffer; cross reads Q [n*l, 256] and K|V [n*s, 512], as engine.loftr_layer does.  Bars: the
    per-element bound of _tol and 5e-3 absolute for the tensor-core route; 2e-5 * max|V| for the FFMA kernel.  Measured on
    a B200 (1 kW power limit): tensor-core route max-abs 2.6e-4, at most 0.075 of the per-element bound; FFMA kernel at most
    0.14 of its bar."""
    c = coarse_cases[case]
    n, l, s = c["shape"]
    C = HEADS * DIM
    dt = torch.float16 if route == "f16" else torch.float32
    flat = lambda x, rows: x.reshape(rows, C)
    if case == "self":
        buf = dev(torch.cat([flat(c["q"], n * l), flat(c["k"], n * s), flat(c["v"], n * s)], 1).to(dt))
        q, k, v, ldq, ldk = buf, buf[:, C:], buf[:, 2 * C:], 3 * C, 3 * C
    else:
        q = dev(flat(c["q"], n * l).to(dt))
        kv = dev(torch.cat([flat(c["k"], n * s), flat(c["v"], n * s)], 1).to(dt))
        k, v, ldq, ldk = kv, kv[:, C:], C, 2 * C
    got = ops.full_attention(q, ldq, k, ldk, v, ldk, n, l, s, HEADS, DIM)
    assert got.dtype == torch.float32 and got.shape == (n * l, C)
    got = got.cpu().view(n, l, HEADS, DIM)
    assert torch.isfinite(got).all()
    worst_abs, worst_ratio = 0.0, 0.0
    for b, r in c["refs"].items():
        err = (got[b, c["rows"]].double() - r["want"]).abs()
        if route == "accurate":
            bar = 2e-5 * r["vabs"]
            assert err.max().item() <= bar, (b, err.max().item(), bar)
            worst_ratio = max(worst_ratio, err.max().item() / bar)
        else:
            ratio = (err / _tol(r)).max().item()
            assert ratio <= 1.0 and err.max().item() <= 5e-3, (b, err.max().item(), ratio)
            worst_ratio = max(worst_ratio, ratio)
        worst_abs = max(worst_abs, err.max().item())
    print(f"[full-attention] coarse {case} {route}: max-abs {worst_abs:.3g}, max err/bar {worst_ratio:.3g}")


# ------------------------------------------------------------------------------------------- B: fine window kernel
@pytest.mark.parametrize("storage", ["f16", "f32"])
@pytest.mark.parametrize("windows", [3, 37, 1003, 112000])
def test_fine_window_full_attention(ops, windows, storage):
    """ops.full_attention_window on the fine self layout (one [m*25, 384] Q|K|V buffer): window m's 25 query rows against
    its own 25 key / value rows, 8 heads x 16.  Logits have a std of ~4 (peaked softmax).  Bar: 1e-5 * max|V| against
    fp64 on the same operands, checked on the first and last 256 windows and 2000 seeded random ones."""
    t, h, d = 25, 8, 16
    c = h * d
    g = torch.Generator(device="cuda").manual_seed(40 + windows)
    x = torch.randn(windows * t, 3 * c, device="cuda", generator=g)
    x[:, :2 * c] *= 2.0
    buf = x.to(torch.float16 if storage == "f16" else torch.float32).contiguous()
    del x
    got = ops.full_attention_window(buf, 3 * c, buf[:, c:], 3 * c, buf[:, 2 * c:], 3 * c, windows, t, h, d)
    assert got.dtype == torch.float32 and got.shape == (windows * t, c)
    gs = torch.Generator().manual_seed(41)
    sel = torch.unique(torch.cat([torch.arange(min(windows, 256)), torch.randint(0, windows, (2000,), generator=gs),
                                  torch.arange(max(0, windows - 256), windows)]))
    rows = (sel[:, None] * t + torch.arange(t)).reshape(-1)
    xs = buf[rows.to(buf.device)].double().cpu().view(len(sel), t, 3, h, d)
    q, k, v = xs[:, :, 0], xs[:, :, 1], xs[:, :, 2]
    want = torch.einsum("mlsh,mshd->mlhd", torch.softmax(torch.einsum("mlhd,mshd->mlsh", q, k) / math.sqrt(d), dim=2), v)
    err = (got[rows.to(got.device)].double().cpu().view(len(sel), t, h, d) - want).abs().max().item()
    bar = 1e-5 * buf[:, 2 * c:].abs().max().item()
    print(f"[full-attention] fine windows={windows} {storage}: max-abs {err:.3g} (bar {bar:.3g})")
    assert err <= bar, (err, bar)


# ------------------------------------------------------------------------------------------- C: one layer vs the oracle
def rnd(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("mode", ["accurate", "shipped"])
def test_full_attention_layers_vs_oracle(ops, mode):
    """engine.loftr_layer / engine.fine_layer with attention='full' (self: x is src; cross: two sequences of different
    lengths at the coarse level) against LF.encoder_layer (LoFTR's FullAttention): 2e-5 of the output range in accurate mode
    (fp32 FFMA kernels), 8e-3 in the shipped configuration (tf32 projections, fp16 Q|K|V, fp16 attention operands) - the
    bars the linear layers meet.  The full and linear layers differ by > 1e-2 on these inputs."""
    from geoformer_b200 import engine
    sd = synth.make_state_dict(7, True)
    tol = 2e-5 if mode == "accurate" else 8e-3
    with ops.precision_scope(**(ACCURATE if mode == "accurate" else SHIPPED)):
        pw = engine.PackedWeights(sd, torch.device("cuda:0"), torch.float16)
        x0, x1 = rnd(2, 300, 256, seed=8), rnd(2, 200, 256, seed=9)
        f0, f1 = rnd(37, 25, 128, seed=10), rnd(37, 25, 128, seed=11)
        xs, fs = x0.cuda(), f0.cuda()
        cases = (
            ("coarse cross", engine.loftr_layer(pw.coarse[1], x0.cuda(), x1.cuda(), 8, attention="full"),
             ("loftr_coarse.layers.1", x0, x1, 8)),
            ("coarse self", engine.loftr_layer(pw.coarse[0], xs, xs, 8, attention="full"), ("loftr_coarse.layers.0", x0, x0, 8)),
            ("fine cross", engine.fine_layer(pw.fine[1], f0.cuda(), f1.cuda(), 8, attention="full"),
             ("loftr_fine.layers.1", f0, f1, 8)),
            ("fine self", engine.fine_layer(pw.fine[0], fs, fs, 8, attention="full"), ("loftr_fine.layers.0", f0, f0, 8)),
        )
        for name, got, (pre, x, src, nh) in cases:
            with torch.no_grad():
                want = LF.encoder_layer(sd, pre, x, src, nh)
                lin = O.encoder_layer(sd, pre, x, src, nh)
            err = (got.cpu() - want).abs().max().item()
            print(f"[full-attention] layer {name} {mode}: max-abs {err:.3g}")
            assert err <= tol * max(1.0, want.abs().max().item()), (name, err)
            assert (want - lin).abs().max().item() > 1e-2, name


# ------------------------------------------------------------------------------------------- D: whole forward
def _model(sd, coarse_thr, backbone):
    from geoformer_b200.model.full_model import GeoFormer
    from geoformer_b200.model.geo_config import default_cfg as geo_cfg
    from geoformer_b200.model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
    cfg = copy.deepcopy(default_cfg)
    cfg["coarse"]["attention"] = cfg["fine"]["attention"] = "full"
    g = dict(geo_cfg)
    g["coarse_thr"] = coarse_thr
    m = GeoFormer(cfg, g)
    m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
    m.backbone_precision = backbone
    m.capture = True
    return m.eval().to("cuda:0")


def _run(model, precision, im0, im1):
    from geoformer_b200 import ops
    with ops.precision_scope(**precision):
        return model({"image0": im0.cuda(), "image1": im1.cuda()})


def _inputs(golden_dir, name):
    if name == "rect":
        return synth.make_state_dict(7, True), synth.make_image(96, 128, 1), synth.make_image(64, 96, 2)
    g = load_golden(golden_dir, name)
    h, w, n, seed0, rnd_norm = [int(v) for v in g["meta"]]
    im0, im1 = synth.make_pairs(n, h, w, str(g["regime"]), seed0)
    return synth.make_state_dict(7, bool(rnd_norm)), im0, im1


@pytest.mark.parametrize("name", ["small_dense", "small_shift", "small_mixed", "rect"])
def test_accurate_forward_full_attention_matches_oracle(golden_dir, name):
    """GeoFormer with coarse.attention = fine.attention = 'full' in accurate mode (fp32 backbone and FFMA kernels) against
    LF.forward (both levels 'full') on the same inputs (the small_* golden pairs and a rectangular pair, L != S):
    b_ids / i_ids / j_ids and mkpts0_f / mkpts1_f identical.  coarse_thr 0 so that every case has coarse matches."""
    sd, im0, im1 = _inputs(golden_dir, name)
    data = _run(_model(sd, 0.0, "fp32"), ACCURATE, im0, im1)
    with torch.no_grad():
        want = LF.forward(sd, im0, im1, dict(coarse_thr=0.0))
    assert want["b_ids"].numel() > 0
    for k in ("b_ids", "i_ids", "j_ids", "mkpts0_f", "mkpts1_f"):
        assert np.array_equal(data[k].cpu().numpy(), want[k].numpy()), k
    lin = O.forward(sd, im0, im1, dict(coarse_thr=0.0))
    print(f"[full-attention] forward {name}: {want['b_ids'].numel()} coarse / {want['mkpts0_f'].shape[0]} fine matches; "
          f"linear route: {lin['b_ids'].numel()} / {lin['mkpts0_f'].shape[0]}")


def _rms_rel(a, b):
    a, b = torch.as_tensor(a).float().cpu(), torch.as_tensor(b).float().cpu()
    return ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()


def test_shipped_forward_full_attention_480x640(golden_dir):
    """The shipped configuration (fp16 tcgen05 backbone, tf32 projections, fp16 attention operands) with both levels
    'full' on the full_shift_rn_480x640 pair: the coarse-transformer outputs within 5e-3 rel-rms of oracle
    LF.local_feature_transformer(..., 'full') on the oracle's backbone features (the linear route measures 8.5e-4;
    measured on a B200: 8.7e-4 / 8.5e-4)."""
    sd, im0, im1 = stage_case_inputs(load_golden(golden_dir, "full_shift_rn_480x640"))
    data = _run(_model(sd, 0.0, "f16"), SHIPPED, im0, im1)
    st = data["_stages"]
    with torch.no_grad():
        c, _ = O.backbone(sd, torch.cat([im0, im1], 0))
        x0, x1 = O.add_pe_flatten(c[:1]), O.add_pe_flatten(c[1:])
        t0, t1 = LF.local_feature_transformer(sd, "loftr_coarse", x0, x1, O.DEFAULT_CFG["coarse_layers"], 8, "full")
    e0, e1 = _rms_rel(st["coarse0"], t0), _rms_rel(st["coarse1"], t1)
    print(f"[full-attention] shipped 480x640 coarse-transformer rel-rms {e0:.3g} / {e1:.3g}; "
          f"{data['mkpts0_f'].shape[0]} fine matches")
    assert max(e0, e1) <= 5e-3, (e0, e1)
    assert data["mkpts0_f"].shape[0] > 0 and torch.isfinite(data["mconf"]).all()
