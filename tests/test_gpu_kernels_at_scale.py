"""GPU parity tests of the product kernels at the batch and shapes bench.py runs (16 pairs at 480x640: 32 images of
4800 tokens, ~4000 anchors per image; 768x768 and 840x840 too).  tests/test_gpu_kernels.py checks every operator at
small shapes; several product kernels change their control flow with batch size, token count or the values themselves,
and those branches only run here:

  A  geo_flash_attn_kernel (flash_attn.cu): the lazy rescale of O and of the row sum, the K / V ring wrapping many times,
     4800-wide anchor lists, a half-empty last query tile, anchor counts 0 / 1 / 65 / 257 / 4000 / 4800;
  B  linattn_partial_mma_kernel / linattn_apply_mma_kernel (linattn.cu): every chunk size the batch-dependent chunking
     picks for the shipped calls, a partial last 32-token slab, the strided Q|K|V layouts of engine.loftr_layer;
  C  gf_coarse_match_fused at batch 16 (CTA pairs decode work items across sample boundaries), exact re-scans included;
  D  the gathers and element-wise kernels of the shipped path that had no direct test.

References are fp64 on the CPU, computed on the same fp16-rounded operands the kernel reads; large ones on a fixed
subset of query rows (rows are independent).  A test that exists to reach a branch also asserts on the host that its
inputs reach it.  Measured numbers quoted in the docstrings: B200, driver-default clocks and power limit (1 kW)."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import geoformer_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from geoformer_b200 import ops as _ops
    assert torch.cuda.is_available(), "GPU tests need a B200"
    _ops.ensure_init(torch.device("cuda:0"))
    return _ops


def dev(t):
    return t.cuda().contiguous()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g) * scale


# ------------------------------------------------------------------------------------------- A: geo flash attention
GEO_N, GEO_L, GEO_HEADS, GEO_DIM = 6, 4800, 4, 64
GEO_CNTS = [4000, 0, 1, 65, 4800, 257]      # many ring wraps, skipped sample, single key, tail of 1, full sequence, tail of 1
KBK, KRING, KLAZY = 64, 4, 8.0               # flash_attn.cu: keys per tile, K / V^T ring stages, lazy window (log2 units)
LOG2E = 1.4426950408889634


def _geo_inputs():
    """Q|K|V [n*l, 768] fp16 (one buffer, read in place as engine.geo_self_layer does) with logits shaped per head.

    Each head has a unit direction u; Q and K are random orthogonal to u, queries get +8u on even rows and -8u on odd rows
    (neighbouring lanes of a warp), and the key of anchor j gets r_h(j) * u, so logit = q.k / 8 = noise +- r_h(j):
      head 0: r = 1.6 per key tile: the '+' rows' maximum climbs and is raised every ~4 tiles (logits up to ~120);
      head 1: r climbs 4.9 logits (7.1 log2 units) over the whole sequence: P approaches 2^8 without a raise;
      head 2: plain random logits;
      head 3: the last anchor spikes 40 logits: a raise by ~58 log2 units in the last tile.
    On the '-' rows the logits fall, so later tiles underflow to fp16 subnormals and zeros."""
    n, l, h, d = GEO_N, GEO_L, GEO_HEADS, GEO_DIM
    g = torch.Generator().manual_seed(20)
    u = torch.randn(h, d, generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    perp = lambda x: x - (x * u).sum(-1, keepdim=True) * u
    q = perp(torch.randn(n, l, h, d, generator=g))
    k = perp(torch.randn(n, l, h, d, generator=g))
    v = torch.randn(n, l, h, d, generator=g)
    sign = 1.0 - 2.0 * (torch.arange(l) % 2).float()
    q = q + 8.0 * sign[None, :, None, None] * u
    aidx = torch.zeros(n, l, dtype=torch.int32)                    # anchor lists as wide as the image (anchor_cap = l)
    for b, cnt in enumerate(GEO_CNTS):
        if cnt == 0:
            continue
        sel = torch.sort(torch.randperm(l, generator=g)[:cnt])[0]
        aidx[b, :cnt] = sel.int()
        tile = (torch.arange(cnt) // KBK).float()
        tiles = (cnt + KBK - 1) // KBK
        ramp = torch.zeros(cnt, h)
        ramp[:, 0] = 1.6 * tile
        ramp[:, 1] = 4.9 * tile / max(tiles - 1, 1)
        ramp[cnt - 1, 3] = 40.0
        k[b, sel] += ramp[:, :, None] * u
    qkv = torch.cat([x.reshape(n * l, h * d) for x in (q, k, v)], 1).half()
    return qkv, aidx, torch.tensor(GEO_CNTS, dtype=torch.int32)


def _geo_rows(l):
    """Checked query rows: the first 128-row tile, the partial last tile and 300 seeded random rows in between."""
    g = torch.Generator().manual_seed(21)
    last = (l - 1) // 128 * 128
    return torch.unique(torch.cat([torch.arange(128), torch.randint(128, last, (300,), generator=g), torch.arange(last, l)]))


def _geo_sample_reference(x, sel, rows):
    """fp64 attention of the checked rows of one sample (x [l, 3, h, d] fp64) plus a replay of the kernel's lazy-maximum
    rule: tile maxima in log2 units against a reference maximum that is raised only on a lead > KLAZY.  Also returns two
    deliberately broken fp64 results of the same recurrence: no rescale at all, and O rescaled but the row sum not."""
    h, d = GEO_HEADS, GEO_DIM
    q, k, v = x[rows, 0], x[sel, 1], x[sel, 2]
    s = torch.einsum("rhd,jhd->rhj", q, k) / math.sqrt(d)
    want = torch.einsum("rhj,jhd->rhd", torch.softmax(s, -1), v)
    cnt = sel.shape[0]
    tiles = (cnt + KBK - 1) // KBK
    s2 = F.pad(s * LOG2E, (0, tiles * KBK - cnt), value=-math.inf).view(len(rows), h, tiles, KBK)
    tm2 = s2.amax(-1)                                                               # [R, h, T]
    m2, raised, lead = torch.empty_like(tm2), torch.zeros_like(tm2, dtype=torch.bool), torch.full_like(tm2, -math.inf)
    m = m2[..., 0] = tm2[..., 0]
    for t in range(1, tiles):
        lead[..., t] = tm2[..., t] - m
        raised[..., t] = lead[..., t] > KLAZY
        m = torch.where(raised[..., t], tm2[..., t], m)
        m2[..., t] = m
    p = torch.exp2(s2 - m2[..., None])                                              # the kernel's P of every tile
    vt = F.pad(v, (0, 0, 0, 0, 0, tiles * KBK - cnt)).view(tiles, KBK, h, d)
    o_t = torch.einsum("rhtj,tjhd->rhtd", p, vt)
    l_t = p.sum(-1)
    w = torch.exp2(m2 - m2[..., -1:])                                               # rescale factors up to the last tile
    exact = (o_t * w[..., None]).sum(2) / (l_t * w).sum(2)[..., None]
    assert (exact - want).abs().max().item() <= 1e-9                                # the replay is the same softmax
    return dict(want=want, vmin=v.amin(0), vmax=v.amax(0), vabs=v.abs().max().item(), tiles=tiles, raised=raised,
                lead=lead, p=p, no_rescale=o_t.sum(2) / l_t.sum(2)[..., None],
                o_only=(o_t * w[..., None]).sum(2) / l_t.sum(2)[..., None])


@pytest.fixture(scope="module")
def geo_case():
    qkv, aidx, cnts = _geo_inputs()
    rows = _geo_rows(GEO_L)
    x = qkv.double().view(GEO_N, GEO_L, 3, GEO_HEADS, GEO_DIM)
    refs = {b: _geo_sample_reference(x[b], aidx[b, :cnt].long(), rows) for b, cnt in enumerate(GEO_CNTS) if cnt}
    return dict(qkv=qkv, aidx=aidx, cnts=cnts, rows=rows, refs=refs)


def _geo_tol(r):
    """Per element: O and l come from the same fp16-rounded P (2^-11 relative each), so the error of O / l is bounded by
    2^-11 * max_i |v_i - out| on top of fp32 round-off: bar 2^-10 * max_i |v_i - want| + 1e-5."""
    spread = torch.maximum(r["vmax"] - r["want"], r["want"] - r["vmin"])
    return 2.0 ** -10 * spread + 1e-5


def _assert_geo_premise(case):
    rows, refs = case["rows"], case["refs"]
    plus = rows % 2 == 0
    r0 = refs[0]
    assert r0["tiles"] > 2 * KRING and refs[4]["tiles"] > 2 * KRING                 # the K / V ring comes round > once
    n_raise = r0["raised"].sum(-1)                                                  # [R, h]
    assert n_raise[plus, 0].min().item() >= 10, n_raise[plus, 0].min()              # head 0 '+' rows: raised many times
    assert n_raise[~plus, 0].max().item() == 0                                      # '-' rows: never
    lead_kept = torch.where(r0["raised"], torch.full_like(r0["lead"], -math.inf), r0["lead"]).amax(-1)
    near = (lead_kept[:, 1] > 6) & (lead_kept[:, 1] <= KLAZY)
    assert near.sum().item() >= 20, near.sum()                                      # head 1: P up to 2^6 .. 2^8, no raise
    assert (r0["raised"][plus, 3, -1]).all()                                        # head 3: the spike raises in the last tile
    assert (r0["p"][~plus, 0, -1].amax(-1) < 2.0 ** -25).all()                      # '-' rows of head 0 underflow fp16
    first = r0["raised"][:128].view(4, 32, GEO_HEADS, -1)                           # the 4 warps of the first query tile
    mixed = first.any(1) & ~first.all(1)
    assert mixed[:, 0].any(-1).all(), "every warp has raised and unraised lanes in the same tile"
    for b, r in refs.items():                                                       # either bug would be caught
        if r["tiles"] == 1:                                                         # a single key tile: nothing to rescale
            continue
        tol = _geo_tol(r)
        for name in ("no_rescale", "o_only"):
            ratio = ((r[name] - r["want"]).abs() / tol).max().item()
            assert ratio > 10, (b, name, ratio)


@pytest.mark.parametrize("route", ["f16_qkv", "f32_qkv", "accurate"])
def test_geo_self_attention_shipped_shape_lazy_rescale(ops, geo_case, route):
    """geo self attention at the shipped shape with the lazy rescale forced (see _geo_inputs), three routes:
    'f16_qkv' (product: fp16 Q|K|V read in place, gf_gather_anchor_kv_h16, gf_geo_self_attention_tc), 'f32_qkv' (fp32 Q|K|V
    holding the same values: gf_gather_anchor_kv_f16 rounds Q, K, V itself) and 'accurate' (gf_geo_self_attention, fp32
    FFMA, online softmax).  Bars: the derived per-element bound of _geo_tol and 5e-3 absolute for the fp16 routes; 2e-5 *
    max|V| for the accurate kernel.  Premise (sample 0, 63 key tiles): every head-0 '+' row is raised 14-16 times, 235 of
    the 486 checked head-1 rows peak at a lead in (6, 8] without a raise, 229 (warp, tile) pairs of the first query tile
    mix raised and unraised lanes; the two broken recurrences miss the bound by 506x and 495x.  Measured on a B200: fp16
    and fp32 routes max-abs 2.9e-4, at most 0.091 of the per-element bound; accurate kernel 1.85e-5 = 0.17 of its bar on
    logits up to 123."""
    _assert_geo_premise(geo_case)
    qkv, aidx, cnts, rows = geo_case["qkv"], geo_case["aidx"], geo_case["cnts"], geo_case["rows"]
    n, l, h, d = GEO_N, GEO_L, GEO_HEADS, GEO_DIM
    c = h * d
    buf = dev(qkv if route == "f16_qkv" else qkv.float())
    got = ops.geo_self_attention(buf, 3 * c, buf[:, c:], 3 * c, buf[:, 2 * c:], 3 * c, n, l, h, d, dev(aidx), dev(cnts),
                                 max_cnt=max(GEO_CNTS), impl="ref" if route == "accurate" else "tf32")
    got = got.cpu().view(n, l, h, d)
    assert torch.isfinite(got).all()
    worst_abs, worst_ratio = 0.0, 0.0
    for b, cnt in enumerate(GEO_CNTS):
        if cnt == 0:
            assert (got[b] == 0).all()
            continue
        r = geo_case["refs"][b]
        err = (got[b, rows].double() - r["want"]).abs()
        if route == "accurate":
            bar = 2e-5 * r["vabs"]
            assert err.max().item() <= bar, (b, err.max().item(), bar)
            worst_ratio = max(worst_ratio, err.max().item() / bar)
        else:
            ratio = (err / _geo_tol(r)).max().item()
            assert ratio <= 1.0 and err.max().item() <= 5e-3, (b, err.max().item(), ratio)
            worst_ratio = max(worst_ratio, ratio)
        worst_abs = max(worst_abs, err.max().item())
    print(f"[at-scale] geo_self {route}: max-abs {worst_abs:.3g}, max err/bar {worst_ratio:.3g}")


# ------------------------------------------------------------------------------------------- B: linear attention
def _chunk_tokens(n, s):
    """gf_linattn_reduce_f16 (linattn.cu): ~600 CTAs whatever the batch, a multiple of 32 tokens in [128, 512]."""
    ct = (s * n // 592 + 31) // 32 * 32
    return min(max(ct, 128), 512)


LINATTN_CASES = [   # (n, l, s, layout) as engine.loftr_layer calls it: self on the 2N-image batch, cross on N pairs
    (32, 4800, 4800, "self"), (16, 4800, 4800, "cross"),           # 480x640
    (32, 9216, 9216, "self"), (16, 9216, 9216, "cross"),           # 768x768
    (32, 11025, 11025, "self"), (16, 11025, 11025, "cross"),       # 840x840
    (16, 4800, 11025, "cross"),                                    # l != s: the apply kernel's partial 64-row tile at the end
]


def test_linattn_cases_cover_every_product_chunking():
    sizes = {_chunk_tokens(n, s) for n, _, s, _ in LINATTN_CASES}
    assert sizes == {160, 256, 288, 320, 512}, sizes
    assert _chunk_tokens(2, 300) == 128                              # test_gpu_kernels.py::test_linear_attention_fp16_storage
    assert any((s % _chunk_tokens(n, s)) % 32 for n, _, s, _ in LINATTN_CASES)     # a partial last 32-token slab
    assert any(l % 64 for _, l, _, _ in LINATTN_CASES)


def _linattn_inputs(n, l, s, layout, seed, dtype=torch.float16):
    """The product's distribution (Q, K = elu+1 of N(0,1), V ~ N(0,1)), generated one sample at a time.
    self: one [n*s, 768] Q|K|V buffer; cross: Q [n*l, 256] and one [n*s, 512] K|V buffer."""
    g = torch.Generator().manual_seed(seed)
    c = 256
    elu1 = lambda rows, cols: F.elu(torch.randn(rows, cols, generator=g)) + 1
    if layout == "self":
        buf = torch.empty(n * s, 3 * c, dtype=dtype)
        for b in range(n):
            buf[b * s:(b + 1) * s, :2 * c] = elu1(s, 2 * c)
            buf[b * s:(b + 1) * s, 2 * c:] = torch.randn(s, c, generator=g)
        return buf, buf
    q, kv = torch.empty(n * l, c, dtype=dtype), torch.empty(n * s, 2 * c, dtype=dtype)
    for b in range(n):
        q[b * l:(b + 1) * l] = elu1(l, c)
        kv[b * s:(b + 1) * s, :c] = elu1(s, c)
        kv[b * s:(b + 1) * s, c:] = torch.randn(s, c, generator=g)
    return q, kv


def _linattn_run(ops, qb, kvb, n, l, s, layout):
    c = 256
    Q = dev(qb)
    KV = Q if layout == "self" else dev(kvb)
    if layout == "self":
        return ops.linattn(Q, 3 * c, KV[:, c:], 3 * c, KV[:, 2 * c:], 3 * c, n, l, s, 8, 32)
    return ops.linattn(Q, c, KV, 2 * c, KV[:, c:], 2 * c, n, l, s, 8, 32)


def _linattn_ref64(q, k, v, heads=8, dim=32):
    """fp64 restatement of linear_attention.py:44-51 on feature-mapped Q, K (as in test_linear_attention_fp16_storage)."""
    l, s = q.shape[0], k.shape[0]
    Q, K, V = (t.double().reshape(-1, heads, dim) for t in (q, k, v))
    KV = torch.einsum("shd,shv->hdv", K, V / s)
    Z = 1 / (torch.einsum("lhd,hd->lh", Q, K.sum(0)) + 1e-6)
    return (torch.einsum("lhd,hdv,lh->lhv", Q, KV, Z) * s).reshape(l, heads * dim)


def _f16_storage_bar(want):
    """fp32-kernel tolerance + one fp16 rounding each of KV, Ksum and the output (test_linear_attention_fp16_storage)."""
    return (2e-5 + 3 * 2.0 ** -11) * max(1.0, want.abs().max().item())


def _linattn_slices(qb, kvb, b, l, s, layout):
    c = 256
    if layout == "self":
        x = qb[b * s:(b + 1) * s]
        return x[:, :c], x[:, c:2 * c], x[:, 2 * c:]
    y = kvb[b * s:(b + 1) * s]
    return qb[b * l:(b + 1) * l], y[:, :c], y[:, c:]


@pytest.mark.parametrize("n,l,s,layout", LINATTN_CASES)
def test_linear_attention_fp16_product_chunkings(ops, n, l, s, layout):
    """fp16-storage linear attention (mma.sync reduce + apply) at every chunk size the shipped calls get, in the strided
    layouts engine.loftr_layer passes; fp64 reference per sample on the same fp16 values.  Measured on a B200: max
    err / bar 0.014-0.019 over the cases (max-abs <= 2.8e-5)."""
    ct = _chunk_tokens(n, s)
    qb, kvb = _linattn_inputs(n, l, s, layout, seed=n + l + s)
    got = _linattn_run(ops, qb, kvb, n, l, s, layout)
    assert got.dtype == torch.float16 and got.shape == (n * l, 256)
    got = got.cpu()
    worst = 0.0
    for b in range(n):
        want = _linattn_ref64(*_linattn_slices(qb, kvb, b, l, s, layout))
        err = (got[b * l:(b + 1) * l].double() - want).abs().max().item()
        bar = _f16_storage_bar(want)
        assert err <= bar, (b, err, bar)
        worst = max(worst, err / bar)
    print(f"[at-scale] linattn f16 n={n} l={l} s={s} {layout} chunk={ct} ({-(-s // ct)} chunks, last slab "
          f"{(s % ct) % 32 or 32} rows): max err/bar {worst:.3g}")


def test_linear_attention_fp32_kernels_long_sequence(ops):
    """fp32 kernels (accurate mode: fixed 256-token chunks, partial last slab of 17 tokens at s = 11025) in the self layout
    against fp64, the 2e-5 bar of test_linear_attention (measured on a B200: 1.9e-8)."""
    n, s = 2, 11025
    assert (s % 256) % 32 == 17
    qb, _ = _linattn_inputs(n, s, s, "self", seed=7, dtype=torch.float32)
    got = _linattn_run(ops, qb, qb, n, s, s, "self").cpu()
    assert got.dtype == torch.float32
    for b in range(n):
        want = _linattn_ref64(*_linattn_slices(qb, qb, b, s, s, "self"))
        err = (got[b * s:(b + 1) * s].double() - want).abs().max().item()
        assert err <= 2e-5 * max(1.0, want.abs().max().item()), (b, err)
        print(f"[at-scale] linattn fp32 s={s} sample {b}: max-abs {err:.3g}")


# ------------------------------------------------------------------------------------------- C: fused matcher, batch 16
def _match_lists(d):
    return torch.stack([d["b_ids"].cpu(), d["i_ids"].cpu(), d["j_ids"].cpu()], 1)


def test_fused_coarse_matching_batch16_shipped_shape(ops):
    """gf_coarse_match_fused at the shipped batch (16 pairs, L = S = 4800, border 2) with flat, peaky and tied samples.
    Samples 0, 7 and 15 carry duplicated f1 rows (exactly equal logit columns) whose earlier copy lies in the border
    strip, so pass 1's smallest-j candidate is rejected and the exact re-scan must recover the later copy - at the first,
    a middle and the last sample of the batch.  (b, i, j) and per-sample counts bit-exact vs the materialised kernels,
    confidences 1e-4 relative (measured on a B200: 22 587 matches, 1.5e-5); samples 0 and 15 bit-exact vs the oracle."""
    n, hw, l, c, border = 16, (60, 80), 4800, 256, 2
    w = hw[1]
    tied = (0, 7, 15)
    f0, f1 = torch.empty(n, l, c), torch.empty(n, l, c)
    for b in range(n):
        rms, off = (1.0, 0.3) if b in tied else ((0.3, 0.1) if b % 2 else (3.0, 1.5))     # tied / flat / peaky
        f0[b] = rnd(l, c, seed=100 + 2 * b, scale=rms) + off
        f1[b] = rnd(l, c, seed=101 + 2 * b, scale=rms) + off
    # (i, j_border, j_inside): f0[i] is aligned with two identical f1 rows; the border copy has the smaller index
    pairs = [(10 * w + 10, 0 * w + 5, 30 * w + 40), (20 * w + 33, 40 * w + 1, 50 * w + 50),
             (45 * w + 70, 0 * w + 70, 44 * w + 44), (57 * w + 3, 25 * w + 79, 33 * w + 7)]
    inside = lambda t: border <= t // w < hw[0] - border and border <= t % w < w - border
    for i, ja, jb in pairs:
        assert ja < jb and not inside(ja) and inside(jb) and inside(i)
        for b in tied:
            f1[b, jb] = f1[b, ja]
            f0[b, i] = 3.0 * f1[b, ja]
    oracle = {}
    for b in (0, n - 1):                                           # the premise: pass 1's candidate fails, re-scan needed
        conf = O.dual_softmax_conf(f0[b:b + 1], f1[b:b + 1], 0.1)
        want = O.coarse_match(conf, 0.0, (hw[0] * 8, hw[1] * 8), hw, hw, border)
        wl = torch.stack([want["i_ids"], want["j_ids"]], 1)
        for i, ja, jb in pairs:
            assert conf[0, i, ja] == conf[0, i, jb] == conf[0, i].max()
            hit = wl[wl[:, 0] == i]
            assert hit.shape[0] == 1 and int(hit[0, 1]) == jb
        oracle[b] = wl
        del conf
    fused, counts = ops.coarse_match_fused(dev(f0), dev(f1), 0.1, 0.0, border, hw, hw, 8.0)
    a = _match_lists(fused)
    sim = ops.similarity(dev(f0), dev(f1), 0.1)
    cf, crmax, ccmax = ops.dual_softmax_(sim)
    mat, counts2 = ops.mutual_nearest(cf, crmax, ccmax, 0.0, border, hw, hw, 8.0)
    del sim, cf
    assert torch.equal(a, _match_lists(mat))
    assert counts.tolist() == counts2.tolist() and (counts > 0).all()
    rel = ((fused["mconf"] - mat["mconf"]).abs() / mat["mconf"].abs().clamp(min=1e-30)).max().item()
    assert rel <= 1e-4, rel
    for b, wl in oracle.items():
        assert torch.equal(a[a[:, 0] == b][:, 1:], wl), b
    print(f"[at-scale] fused matcher batch 16: {a.shape[0]} matches, counts {counts.tolist()}, conf rel {rel:.3g}")


# ------------------------------------------------------------------------------------------- D: gathers, element-wise
def _fine_gather_check(ops, fmap16, b_ids, tok, wc, stride, out_dtype, chunk=16384):
    """gf_fine_gather_f16 / gf_fine_gather_f16_f16 (NHWC fp16 map) vs O.fine_windows on the map's fp16 values, bit-exact;
    the output is pre-filled with NaN so that an element the kernel skips cannot pass."""
    m, c = b_ids.shape[0], fmap16.shape[1]
    out = torch.full((m, 25, c), math.nan, dtype=out_dtype).cuda()
    got = ops.fine_gather(dev(fmap16.permute(0, 2, 3, 1)), dev(b_ids), dev(tok), wc, stride, 5, out=out)
    assert got.dtype == out_dtype and got.shape == (m, 25, c)
    got = got.cpu()
    ref = fmap16.float()
    for a in range(0, m, chunk):
        want = O.fine_windows(ref, b_ids[a:a + chunk], tok[a:a + chunk], 5, stride)
        assert torch.equal(got[a:a + chunk].float(), want), a


@pytest.mark.parametrize("out_dtype", [torch.float32, torch.float16])
def test_fine_gather_from_fp16_map(ops, out_dtype):
    """The backbone's fp16 fine map -> fp32 windows (gf_fine_gather_f16) and fp16 windows (gf_fine_gather_f16_f16):
    corner and edge tokens (zero padding), w_c != h_c, several samples, m = 0, and the shipped batch's ~56 000 fine
    matches (one CTA per match) on a 240 x 320 map."""
    g = torch.Generator().manual_seed(30)
    n, c, hc, wc, st = 3, 128, 12, 17, 4
    fmap = rnd(n, c, hc * st, wc * st, seed=31).half()
    m = 300
    b_ids, tok = torch.randint(0, n, (m,), generator=g), torch.randint(0, hc * wc, (m,), generator=g)
    edge = [0, wc - 1, (hc - 1) * wc, hc * wc - 1, 5, (hc - 1) * wc + 7, 4 * wc, 7 * wc - 1, wc + 1, (hc - 2) * wc + wc - 2]
    tok[:len(edge)] = torch.tensor(edge)
    b_ids[:len(edge)] = torch.arange(len(edge)) % n
    _fine_gather_check(ops, fmap, b_ids, tok, wc, st, out_dtype)
    _fine_gather_check(ops, fmap, b_ids[:0], tok[:0], wc, st, out_dtype)
    n, hc, wc, m = 2, 60, 80, 56000
    fmap = rnd(n, c, hc * st, wc * st, seed=32).half()
    b_ids, tok = torch.randint(0, n, (m,), generator=g), torch.randint(0, hc * wc, (m,), generator=g)
    tok[:4] = torch.tensor([0, wc - 1, (hc - 1) * wc, hc * wc - 1])
    _fine_gather_check(ops, fmap, b_ids, tok, wc, st, out_dtype)


def test_gather_rows_shipped_batch(ops):
    """gf_gather_rows (coarse context rows of the fine stage) into both halves of one buffer, as engine.fine_stage does."""
    n, l, c, m = 16, 4800, 256, 56000
    g = torch.Generator().manual_seed(33)
    feat = rnd(n, l, c, seed=34)
    b_ids, tok = torch.randint(0, n, (m,), generator=g), torch.randint(0, l, (m,), generator=g)
    b_ids[:4], tok[:4] = torch.tensor([0, 0, n - 1, n - 1]), torch.tensor([0, l - 1, 0, l - 1])
    ctx = torch.full((2 * m, c), math.nan).cuda()
    fd, bd = dev(feat), dev(b_ids)
    ops.gather_rows(fd, bd, dev(tok), out=ctx[:m])
    ops.gather_rows(fd, bd, dev(tok.flip(0)), out=ctx[m:])
    got = ctx.cpu()
    assert torch.equal(got[:m], feat[b_ids, tok]) and torch.equal(got[m:], feat[b_ids, tok.flip(0)])


def test_select_rows_keeps_flagged_samples(ops):
    """gf_select_rows: samples with flag 0 get src, every other sample of dst is left untouched (sentinel)."""
    n, l, c = 16, 4800, 256
    src = rnd(n * l, c, seed=35)
    flag = torch.tensor([0, 1, 4000, 0, -1, 0, 0, 7, 1, 0, 4800, 0, 0, 2, 0, 0], dtype=torch.int32)
    dst = torch.full((n * l, c), -12345.0).cuda()
    ops.select_rows_(dst, dev(src), dev(flag), n, l, c)
    got, src = dst.cpu().view(n, l, c), src.view(n, l, c)
    for b in range(n):
        assert torch.equal(got[b], src[b]) if flag[b] == 0 else (got[b] == -12345.0).all(), b


def test_add_posenc_bit_exact(ops):
    """gf_add_posenc on the 2N-image batch: x + pe in fp32, bit-exact."""
    n, l, c = 32, 4800, 256
    x, pe = rnd(n, l, c, seed=36), O.position_encoding(c, 60, 80).reshape(c, l).t().contiguous()
    got = ops.add_posenc(dev(x), dev(pe)).cpu()
    assert torch.equal(got, x + pe)
