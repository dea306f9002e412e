"""The drop-in boundary (SURVEY.md §8b, a16): the reference's matcher wrappers run on top of this repo's `model.*`
modules with ONE added line — ``sys.path.insert(0, "<repo>/geoformer_b200")`` (INTEGRATION.md §1).

* CPU: a fresh interpreter with that line only executes the wrapper's three import statements
  (eval_tool/immatch/modules/geoformer.py:6-10) and its ctor/load sequence (:23-31).  When GEOFORMER_REFERENCE names a
  checkout of the reference repository, the UNMODIFIED wrapper class itself is constructed on top of the drop-in modules.
* GPU: `match_inputs_` (:50-54,73) and `match_pairs` (:77-99) run through the top-level `model.*` imports on image
  files; the matches are compared with the CPU oracle on the same resized tensors.  Without a reference checkout the
  wrapper is the restatement below (same statements, same order).
"""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "geoformer_b200")
REFERENCE = os.environ.get("GEOFORMER_REFERENCE", "")      # optional checkout of the reference repository

# what a maintainer adds on top of eval_Hpatches.py / eval_FIRE.py / eval_ISC.py / inference.py
INTEGRATION_LINE = f"import sys; sys.path.insert(0, {DROPIN!r})"

# arithmetic-free stand-ins for third-party packages the reference imports but this image lacks (SURVEY.md §8c)
STUBS = textwrap.dedent("""
    import sys, types
    def _stub(name, **attrs):
        m = types.ModuleType(name); m.__dict__.update(attrs); sys.modules[name] = m
    for _n in ("skimage", "kornia", "kornia.geometry", "kornia.utils", "imgaug", "pydegensac", "yacs"):
        _stub(_n)
    _stub("skimage.feature", peak_local_max=None); _stub("kornia.geometry.subpix", dsnt=None)
    _stub("kornia.utils.grid", create_meshgrid=None); _stub("imgaug.augmenters"); _stub("yacs.config", CfgNode=dict)
    sys.modules["imgaug"].augmenters = sys.modules["imgaug.augmenters"]
""")


def _run(code: str, cwd: str):
    env = {k: v for k, v in os.environ.items() if k != "PYTHONPATH"}     # the repo root must NOT be importable a priori
    r = subprocess.run([sys.executable, "-c", code], cwd=cwd, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, f"stdout:\n{r.stdout}\nstderr:\n{r.stderr}"
    return r.stdout


def _save_ckpt(path):
    from geoformer_b200 import synth
    torch.save({"state_dict": {"matcher." + k: v for k, v in synth.make_state_dict(0).items()}}, path)


def test_wrapper_imports_and_ctor_sequence_from_a_foreign_cwd(tmp_path):
    """geoformer.py:6-10 + :23-31 in a fresh interpreter whose only knowledge of this repo is the INTEGRATION.md line."""
    ckpt = str(tmp_path / "geoformer.ckpt")
    _save_ckpt(ckpt)
    code = INTEGRATION_LINE + textwrap.dedent(f"""
        import torch
        from model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
        from model.full_model import GeoFormer as GeoFormer_
        from model.geo_config import default_cfg as geoformer_cfg
        conf = dict(default_cfg)
        conf['match_coarse']['thr'] = 0.35
        geoformer_cfg['coarse_thr'] = 0.35
        model = GeoFormer_(conf)
        ckpt_dict = torch.load({ckpt!r}, map_location=torch.device('cpu'))
        if 'state_dict' in ckpt_dict:
            ckpt_dict = ckpt_dict['state_dict']
        res = model.load_state_dict(ckpt_dict, strict=False)
        model = model.eval().to(torch.device('cpu'))
        assert not res.missing_keys and not res.unexpected_keys, res
        assert len(model.state_dict()) == 253
        assert model.geo_cfg is geoformer_cfg and model.geo_cfg['coarse_thr'] == 0.35
        assert model.config['match_coarse']['thr'] == 0.35 and default_cfg['match_coarse']['thr'] == 0.35
        import model.full_model as fm
        assert fm.__file__.startswith({DROPIN!r}), fm.__file__
        try:                                        # no CPU fallback: a CPU forward must fail loudly
            model({{'image0': torch.zeros(1, 1, 64, 64), 'image1': torch.zeros(1, 1, 64, 64)}})
        except RuntimeError as e:
            assert 'CUDA' in str(e)
        else:
            raise SystemExit('CPU forward did not raise')
        print('DROPIN-OK')
    """)
    assert "DROPIN-OK" in _run(code, cwd=str(tmp_path))


@pytest.mark.skipif(not os.path.isdir(REFERENCE), reason="needs GEOFORMER_REFERENCE: a checkout of the reference repository")
def test_unmodified_reference_wrapper_constructs_on_the_dropin(tmp_path):
    """The real `eval_tool.immatch.modules.geoformer.GeoFormer` (imported from the reference checkout, unmodified) builds its
    model from THIS repo's `model.*` and loads a checkpoint-shaped file through its own ctor."""
    ckpt = str(tmp_path / "geoformer.ckpt")
    _save_ckpt(ckpt)
    code = STUBS + INTEGRATION_LINE + textwrap.dedent(f"""
        sys.path.insert(1, {REFERENCE!r})           # the script's own directory, as when eval_Hpatches.py is run in place
        from eval_tool.immatch.modules.geoformer import GeoFormer
        w = GeoFormer(dict(imsize=480, match_threshold=0.2, no_match_upscale=False, ckpt={ckpt!r}))
        import model.full_model as fm, inspect
        assert fm.__file__.startswith({DROPIN!r}), fm.__file__
        assert type(w.model) is fm.GeoFormer and not w.model.training
        assert inspect.getsourcefile(type(w)).startswith({REFERENCE!r})
        assert w.model.geo_cfg['coarse_thr'] == 0.2 and w.model.config['match_coarse']['thr'] == 0.2
        assert w.name == 'GeoFormer_geoformer'
        print('WRAPPER-OK')
    """)
    assert "WRAPPER-OK" in _run(code, cwd=str(tmp_path))


# ------------------------------------------------------------------------------------------------ GPU
WRAPPER_RESTATEMENT = textwrap.dedent("""
    # eval_tool/immatch/modules/geoformer.py:12-99 + utils/data_io.py:16-26,48-62, statement for statement
    import cv2, numpy as np, torch
    from argparse import Namespace
    from model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
    from model.full_model import GeoFormer as GeoFormer_
    from model.geo_config import default_cfg as geoformer_cfg

    def resize_im(wo, ho, imsize=None, dfactor=1, value_to_scale=max):
        wt, ht = wo, ho
        if imsize and value_to_scale(wo, ho) > imsize and imsize > 0:
            scale = imsize / value_to_scale(wo, ho)
            ht, wt = int(round(ho * scale)), int(round(wo * scale))
        wt, ht = map(lambda x: int(x // dfactor * dfactor), [wt, ht])
        return wt, ht, (wo / wt, ho / ht)

    class GeoFormer:
        def __init__(self, args, gpuid=0):
            self.device = torch.device('cuda:{}'.format(gpuid) if torch.cuda.is_available() else 'cpu')
            torch.set_grad_enabled(False)
            args = Namespace(**args) if type(args) == dict else args
            self.imsize, self.match_threshold, self.no_match_upscale = args.imsize, args.match_threshold, args.no_match_upscale
            conf = dict(default_cfg)
            conf['match_coarse']['thr'] = self.match_threshold
            geoformer_cfg['coarse_thr'] = self.match_threshold
            self.model = GeoFormer_(conf)
            ckpt_dict = torch.load(args.ckpt, map_location=torch.device('cpu'))
            if 'state_dict' in ckpt_dict:
                ckpt_dict = ckpt_dict['state_dict']
            self.model.load_state_dict(ckpt_dict, strict=False)
            self.model = self.model.eval().to(self.device)

        def load_im(self, im_path):
            im = cv2.imread(im_path, cv2.IMREAD_GRAYSCALE)
            ho, wo = im.shape
            wt, ht, scale = resize_im(wo, ho, imsize=self.imsize, dfactor=8, value_to_scale=min)
            im = cv2.resize(im, (wt, ht))
            return torch.from_numpy(im).float().div(255)[None, None].to(self.device), scale

        def match_inputs_(self, gray1, gray2):
            batch = {'image0': gray1, 'image1': gray2}
            with torch.no_grad():
                batch = self.model(batch)
            kpts1 = batch['mkpts0_f'].cpu().numpy()
            kpts2 = batch['mkpts1_f'].cpu().numpy()
            scores = batch['mconf'].cpu().numpy()
            return np.concatenate([kpts1, kpts2], axis=1), kpts1, kpts2, scores

        def match_pairs(self, im1_path, im2_path):
            torch.cuda.empty_cache()
            gray1, sc1 = self.load_im(im1_path)
            gray2, sc2 = self.load_im(im2_path)
            upscale = np.array([sc1 + sc2])
            matches, kpts1, kpts2, scores = self.match_inputs_(gray1, gray2)
            if self.no_match_upscale:
                return matches, kpts1, kpts2, scores, upscale.squeeze(0)
            return upscale * matches, sc1 * kpts1, sc2 * kpts2, scores
""")


@pytest.mark.gpu
def test_match_pairs_through_toplevel_model_imports(tmp_path):
    """Wrapper call sequence on image files, in a fresh interpreter that knows this repo only through the
    INTEGRATION.md line; result vs the CPU oracle on the same resized tensors (the unmodified reference wrapper is used
    when a reference checkout is given, the restatement above otherwise)."""
    import cv2
    from geoformer_b200 import synth
    from oracle import geoformer_oracle as O
    ckpt = str(tmp_path / "geoformer.ckpt")
    _save_ckpt(ckpt)
    rng = np.random.RandomState(5)
    im = rng.randint(0, 256, (240, 320)).astype(np.uint8)         # min side 240 > imsize 96 -> resized to 128x96
    p0, p1 = str(tmp_path / "a.png"), str(tmp_path / "b.png")
    cv2.imwrite(p0, im); cv2.imwrite(p1, im)
    out = str(tmp_path / "out.npz")
    if os.path.isdir(REFERENCE):
        head = STUBS + INTEGRATION_LINE + f"\nsys.path.insert(1, {REFERENCE!r})\n" \
            "from eval_tool.immatch.modules.geoformer import GeoFormer\nimport numpy as np, torch\n"
    else:
        head = INTEGRATION_LINE + WRAPPER_RESTATEMENT
    code = head + textwrap.dedent(f"""
        w = GeoFormer(dict(imsize=96, match_threshold=0.0, no_match_upscale=False, ckpt={ckpt!r}))
        assert w.device.type == 'cuda'
        matches, k1, k2, scores = w.match_pairs({p0!r}, {p1!r})
        w.no_match_upscale = True
        m2, r1, r2, s2, up = w.match_pairs({p0!r}, {p1!r})
        g1, sc1 = w.load_im({p0!r})
        import model.full_model as fm
        assert fm.__file__.startswith({DROPIN!r})
        np.savez({out!r}, matches=matches, k1=k1, k2=k2, scores=scores, m2=m2, r1=r1, r2=r2, s2=s2, up=up,
                 gray=g1.cpu().numpy(), sc=np.asarray(sc1))
        print('MATCH-OK', matches.shape)
    """)
    assert "MATCH-OK" in _run(code, cwd=str(tmp_path))
    z = np.load(out)
    assert z["gray"].shape == (1, 1, 96, 128) and np.allclose(z["sc"], [2.5, 2.5])
    assert z["matches"].shape[1] == 4 and z["matches"].shape[0] == z["scores"].shape[0] > 20
    assert z["matches"].dtype == np.float64 or z["matches"].dtype == np.float32
    assert np.array_equal(z["m2"], np.concatenate([z["r1"], z["r2"]], 1)) and np.allclose(z["up"], [2.5, 2.5, 2.5, 2.5])
    assert np.allclose(z["matches"], z["m2"] * 2.5) and np.allclose(z["k1"], z["r1"] * 2.5)
    # same resized tensor through the CPU oracle: >= 90 % of its matches reproduced exactly
    gray = torch.from_numpy(z["gray"])
    with torch.no_grad():
        want = O.forward(synth.make_state_dict(0), gray, gray, dict(coarse_thr=0.0))
    ref = {tuple(r) for r in torch.cat([want["mkpts0_f"], want["mkpts1_f"]], 1).long().tolist()}
    got = {tuple(int(v) for v in r) for r in z["m2"]}
    assert len(got & ref) >= 0.9 * len(ref), (len(got), len(ref), len(got & ref))
