"""Full softmax attention (`attention: 'full'`) on one B200: the coarse d = 32 flash kernel against the d = 64 geo kernel
in the same process (time, exponentials per second: both issue one MUFU exponential per score), and a whole forward at
480x640, batch 16, with 'full' at both levels against the default (linear) configuration.

    python tools/prof_full_attn.py [--out results.json] [--iters 20] [--steps 5]

Kernel times are CUDA events around `iters` back-to-back launches on inputs that were laid out once (K / V^T tiles of
157 / 79 MB per call for d = 32: larger than L2).  Forward steps alternate the two configurations."""
import argparse
import copy
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from geoformer_b200 import _lib, ops, synth


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def events(fn, iters):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels(iters):
    dev = torch.device("cuda:0")
    g = torch.Generator(device="cuda").manual_seed(0)
    s32 = lambda: torch.cuda.current_stream().cuda_stream
    # d = 32: LoFTR coarse self attention, 16 pairs at 480x640 (32 images x 4800 tokens), 8 heads
    n, l, h, d = 32, 4800, 8, 32
    c = h * d
    qkv = (torch.randn(n * l, 3 * c, device=dev, generator=g) * 0.5).half()
    s_pad = (l + 63) // 64 * 64
    kg = torch.empty((h, n, s_pad, d), device=dev, dtype=torch.float16)
    vt = torch.empty((h, n, d, s_pad), device=dev, dtype=torch.float16)
    cnt = torch.empty(n, device=dev, dtype=torch.int32)
    out = torch.empty((n * l, c), device=dev)
    _lib.call("gf_dense_kv_h16", qkv[:, c:].data_ptr(), 3 * c, qkv[:, 2 * c:].data_ptr(), 3 * c, n, l, h, d, s_pad,
              kg.data_ptr(), vt.data_ptr(), cnt.data_ptr(), s32())
    t32 = events(lambda: _lib.call("gf_full_attention_tc", qkv.data_ptr(), 3 * c, kg.data_ptr(), vt.data_ptr(), cnt.data_ptr(),
                                   out.data_ptr(), n, l, l, h, d, s_pad, s32()), iters)
    t32_op = events(lambda: ops.full_attention(qkv, 3 * c, qkv[:, c:], 3 * c, qkv[:, 2 * c:], 3 * c, n, l, l, h, d), iters)
    e32 = n * h * l * l
    # d = 64: geo self attention over 4000 anchors per image (the benchmark's regime), 4 heads
    h64, d64, acnt = 4, 64, 4000
    c64 = h64 * d64
    qkv64 = (torch.randn(n * l, 3 * c64, device=dev, generator=g) * 0.5).half()
    aidx = torch.stack([torch.sort(torch.randperm(l, device=dev, generator=g)[:acnt])[0] for _ in range(n)]).int().contiguous()
    cnts = torch.full((n,), acnt, device=dev, dtype=torch.int32)
    s_pad64 = (acnt + 63) // 64 * 64
    kg64 = torch.empty((h64, n, s_pad64, d64), device=dev, dtype=torch.float16)
    vt64 = torch.empty((h64, n, d64, s_pad64), device=dev, dtype=torch.float16)
    out64 = torch.empty((n * l, c64), device=dev)
    _lib.call("gf_gather_anchor_kv_h16", qkv64[:, c64:].data_ptr(), 3 * c64, qkv64[:, 2 * c64:].data_ptr(), 3 * c64, n, l, h64,
              d64, aidx.data_ptr(), cnts.data_ptr(), aidx.shape[1], s_pad64, kg64.data_ptr(), vt64.data_ptr(), s32())
    t64 = events(lambda: _lib.call("gf_geo_self_attention_tc", qkv64.data_ptr(), 3 * c64, kg64.data_ptr(), vt64.data_ptr(),
                                   out64.data_ptr(), n, l, h64, d64, s_pad64, cnts.data_ptr(), s32()), iters)
    e64 = n * h64 * l * acnt
    r = dict(d32_ms=t32, d32_with_relayout_ms=t32_op, d32_exp=e32, d32_exp_per_s=e32 / (t32 * 1e-3),
             d64_ms=t64, d64_exp=e64, d64_exp_per_s=e64 / (t64 * 1e-3))
    r["exp_rate_ratio_d32_over_d64"] = r["d32_exp_per_s"] / r["d64_exp_per_s"]
    return r


def forwards(steps):
    from geoformer_b200.model.full_model import GeoFormer
    from geoformer_b200.model.geo_config import default_cfg as geo_cfg
    from geoformer_b200.model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
    sd = synth.make_state_dict(0)
    im0, im1 = synth.make_pairs(16, 480, 640, "dense", 0)
    im0, im1 = im0.cuda(), im1.cuda()
    models = {}
    for kind in ("linear", "full"):
        cfg = copy.deepcopy(default_cfg)
        cfg["coarse"]["attention"] = cfg["fine"]["attention"] = kind
        g = dict(geo_cfg)
        g["coarse_thr"] = 0.0
        m = GeoFormer(cfg, g)
        m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
        models[kind] = m.eval().to("cuda:0")
    times = {k: [] for k in models}
    matches = {}
    for kind, m in models.items():                                     # warm-up (packing, first launches)
        for _ in range(2):
            matches[kind] = int(m({"image0": im0, "image1": im1})["mkpts0_f"].shape[0])
    for _ in range(steps):
        for kind, m in models.items():
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m({"image0": im0, "image1": im1})
            e1.record(); torch.cuda.synchronize()
            times[kind].append(e0.elapsed_time(e1))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    return dict(forward_ms_median={k: round(v, 2) for k, v in med.items()}, forward_ms_all=times,
                full_minus_linear_ms=med["full"] - med["linear"], fine_matches=matches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_full_attn.py measures on the GPU; no CUDA device found")
    ops.ensure_init(torch.device("cuda:0"))
    name, pl = card()
    res = dict(device=name, power_limit=pl, **kernels(a.iters))
    print(f"{name}, power limit {pl}")
    print(f"d=32 full attention (32 x 4800 x 4800, 8 heads): {res['d32_ms']:.3f} ms kernel "
          f"({res['d32_with_relayout_ms']:.3f} ms with the K / V^T relayout), {res['d32_exp_per_s']:.3e} exp/s")
    print(f"d=64 geo attention  (32 x 4800 x 4000, 4 heads): {res['d64_ms']:.3f} ms kernel, {res['d64_exp_per_s']:.3e} exp/s")
    print(f"exp rate d32 / d64: {res['exp_rate_ratio_d32_over_d64']:.3f}")
    res.update(forwards(a.steps))
    print(f"forward 480x640 batch 16, median ms: {res['forward_ms_median']} (full - linear: {res['full_minus_linear_ms']:.2f} ms)")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)


if __name__ == "__main__":
    main()
