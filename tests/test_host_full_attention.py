"""LoFTR full attention (`coarse.attention` / `fine.attention` = 'full') on CPU: the host path on the emulated operators
(tests/emu_ops.py + tests/emu_ops_full.py) against the checker of tests/loftr_full_oracle.py, the route each
configuration takes, the config values GeoFormer refuses rather than ignores, and tests/test_gpu_full_attention.py run on the emulations (its host logic, premises and fp64 references;
the shipped-shape kernel cases and the 480x640 forward are left to the GPU)."""
import copy
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from geoformer_b200 import ops, synth
from oracle import geoformer_oracle as O
from tests import emu_ops_full as emu
from tests import loftr_full_oracle as LF
from tests.test_host_emulation_contracts import ROOT, emulated_copy
from tests.util import load_golden

ACCURATE = dict(linear="ref", similarity="ref", attention="ref", activations="f32")
SHIPPED = dict(linear="tf32", similarity="f16x3", attention="tf32", activations="f16")


def _cfgs(coarse="linear", fine="linear"):
    from geoformer_b200.model.geo_config import default_cfg as geo_cfg
    from geoformer_b200.model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
    cfg = copy.deepcopy(default_cfg)
    cfg["coarse"]["attention"], cfg["fine"]["attention"] = coarse, fine
    return cfg, dict(geo_cfg)


def _model(monkeypatch, sd, coarse, fine, backbone):
    from geoformer_b200.model.full_model import GeoFormer
    emu.install(monkeypatch)
    cfg, g = _cfgs(coarse, fine)
    g["coarse_thr"] = 0.0
    m = GeoFormer(cfg, g)
    m.load_state_dict({k: v.clone() for k, v in sd.items()}, strict=True)
    m.backbone_precision = backbone
    m.capture = True
    return m.eval()


def _forward(m, precision, im0, im1):
    with ops.precision_scope(**precision), torch.no_grad():
        return m._forward({"image0": im0, "image1": im1}, im0, im1)     # forward() itself refuses CPU tensors


@pytest.mark.parametrize("name", ["small_dense", "small_mixed"])
def test_full_attention_host_path_matches_oracle(monkeypatch, golden_dir, name):
    """Both levels 'full', accurate configuration, emulated operators: the integer outputs equal the checker's forward
    (LF.forward) with the same config, and the attention of every LoFTR layer ran through the full-attention operators
    (coarse: 8 layers, both images; fine: 2 layers, per-op path, never the fused fine-layer kernel)."""
    g = load_golden(golden_dir, name)
    h, w, n, seed0, rnd = [int(v) for v in g["meta"]]
    sd = synth.make_state_dict(7, bool(rnd))
    im0, im1 = synth.make_pairs(n, h, w, str(g["regime"]), seed0)
    d = _forward(_model(monkeypatch, sd, "full", "full", "fp32"), ACCURATE, im0, im1)
    want = LF.forward(sd, im0, im1, dict(coarse_thr=0.0))
    assert want["b_ids"].numel() > 0
    for k in ("b_ids", "i_ids", "j_ids", "mkpts0_f", "mkpts1_f"):
        assert np.array_equal(d[k].numpy(), want[k].numpy()), k
    # same-size pair: coarse self layers run both images as one batch (1 call), cross layers one call per direction
    assert emu.CALLS.get("full_attention", 0) == 4 * 1 + 4 * 2
    assert emu.CALLS.get("full_attention_window", 0) == 1 + 2
    assert emu.CALLS.get("linattn", 0) == 0 and emu.CALLS.get("linattn_window", 0) == 0
    assert emu.CALLS.get("fine_layer_fused", 0) == 0


@pytest.mark.parametrize("coarse,fine", [("linear", "linear"), ("full", "linear"), ("linear", "full")])
def test_each_level_takes_its_configured_route(monkeypatch, coarse, fine):
    """Shipped configuration, emulated operators: the default config never calls the new operators (and keeps the fused
    fine-layer kernel); each level switches on its own key."""
    sd = synth.make_state_dict(7, True)
    im0, im1 = synth.make_pairs(1, 96, 128, "dense", 0)
    d = _forward(_model(monkeypatch, sd, coarse, fine, "f16"), SHIPPED, im0, im1)
    assert d["b_ids"].numel() > 0
    calls = emu.CALLS
    assert (calls.get("full_attention", 0) > 0) == (coarse == "full")
    assert (calls.get("linattn", 0) > 0) == (coarse == "linear")
    assert (calls.get("full_attention_window", 0) > 0) == (fine == "full")
    assert (calls.get("fine_layer_fused", 0) > 0) == (fine == "linear")
    assert calls.get("linattn_window", 0) == 0


def test_unsupported_config_values_are_refused():
    """Config values that would change the result if ignored: an attention kind other than 'linear' / 'full', Sinkhorn
    matching (needs bin_score, not in the checkpoint schema), fine_concat_coarse_feat=False, and coarse full attention
    with padding masks (a fully padded query row is a softmax over -inf only in the reference)."""
    from geoformer_b200.model.full_model import GeoFormer
    for level in ("coarse", "fine"):
        cfg, g = _cfgs()
        cfg[level]["attention"] = "performer"
        with pytest.raises(ValueError):
            GeoFormer(cfg, g)
    cfg, g = _cfgs()
    cfg["match_coarse"]["match_type"] = "sinkhorn"
    with pytest.raises(NotImplementedError):
        GeoFormer(cfg, g)
    cfg, g = _cfgs()
    cfg["fine_concat_coarse_feat"] = False
    with pytest.raises(NotImplementedError):
        GeoFormer(cfg, g)
    m = GeoFormer(*_cfgs("full", "linear")).eval()
    x, mask = torch.zeros(1, 1, 32, 32), torch.ones(1, 4, 4, dtype=torch.bool)
    with pytest.raises(NotImplementedError):
        m({"image0": x, "image1": x, "mask0": mask, "mask1": mask})
    GeoFormer(*_cfgs("full", "full"))                                 # both supported kinds construct


def test_checker_forward_is_the_oracle_forward_with_linear_attention():
    """tests/loftr_full_oracle.forward restates oracle.forward's steps: with linear attention at both levels it gives the
    oracle's integer outputs and coarse features exactly, so only the attention differs on the 'full' route."""
    sd = synth.make_state_dict(7, True)
    im0, im1 = synth.make_pairs(2, 96, 128, "dense", 0)
    with torch.no_grad():
        got = LF.forward(sd, im0, im1, dict(coarse_thr=0.0), coarse="linear", fine="linear")
        want = O.forward(sd, im0, im1, dict(coarse_thr=0.0))
    assert want["mkpts0_f"].shape[0] > 0
    for k in ("b_ids", "i_ids", "j_ids", "mkpts0_c", "mkpts0_f", "mkpts1_f", "mconf"):
        assert torch.equal(got[k], want[k]), k


def test_full_attention_gpu_tests_pass_on_emulated_operators(tmp_path):
    dst = str(tmp_path / "emulated_test_gpu_full_attention.py")
    emulated_copy(os.path.join(ROOT, "tests", "test_gpu_full_attention.py"), dst)
    src = open(dst).read()
    assert src.count("from tests import emu_ops\n") == 1
    open(dst, "w").write(src.replace("from tests import emu_ops\n", "from tests import emu_ops_full as emu_ops\n"))
    r = subprocess.run([sys.executable, "-m", "pytest", dst, "-q", "--no-header", "-p", "no:cacheprovider", "-p", "tests.conftest",
                        "--rootdir", str(tmp_path), "-k", "not shipped_shape and not 112000 and not 480x640"],
                       capture_output=True, text=True, cwd=ROOT, timeout=1500)
    tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-2000:]
    assert r.returncode == 0, r.stdout[-6000:]
    assert " passed" in tail and "failed" not in tail and "error" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 13, tail
