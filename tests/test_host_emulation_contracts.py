"""The operator emulations of tests/emu_ops.py are held to the SAME expectations as the CUDA kernels: the kernel-by-kernel
GPU parity tests (tests/test_gpu_kernels.py — every operator against the CPU oracle, integer outputs bit-exact) are run
here against the emulations, on CPU.  Kernel == oracle (GPU run) and emulation == oracle (this run) on the same cases,
same argument contracts and same tolerances is what makes the host-path tests on emulated operators
(tests/test_host_forward_emulated.py, the bench dry run) meaningful."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

HEADER = '''
import sys
sys.path.insert(0, %r)
import pytest as _pt, torch as _t
@_pt.fixture(autouse=True)
def _emulated_operators(monkeypatch):
    from tests import emu_ops
    emu_ops.install(monkeypatch)
    monkeypatch.setattr(_t.cuda, "is_available", lambda: True)
    monkeypatch.setattr(_t.cuda, "synchronize", lambda *a, **k: None)
    from geoformer_b200.model.full_model import GeoFormer          # forward() itself refuses CPU tensors
    monkeypatch.setattr(GeoFormer, "forward", lambda self, data: self._forward(data, data["image0"], data["image1"]))
''' % ROOT


def emulated_copy(src_path: str, dst_path: str) -> None:
    """A GPU test module with its device strings pointed at the CPU and the operators emulated (nothing else changes)."""
    s = open(src_path).read()
    s = s.replace(".cuda()", ".cpu()").replace('"cuda:0"', '"cpu"').replace('device="cuda"', 'device="cpu"').replace('"cuda"', '"cpu"')
    assert "pytestmark = pytest.mark.gpu" in s
    s = s.replace("pytestmark = pytest.mark.gpu", HEADER)
    s = s.replace('    assert torch.cuda.is_available(), "GPU tests need a B200"\n', "")
    s = s.replace('    _ops.ensure_init(torch.device("cpu"))\n', "")
    open(dst_path, "w").write(s)


def test_emulations_pass_the_kernel_parity_tests(tmp_path):
    dst = str(tmp_path / "emulated_test_gpu_kernels.py")
    emulated_copy(os.path.join(ROOT, "tests", "test_gpu_kernels.py"), dst)
    r = subprocess.run([sys.executable, "-m", "pytest", dst, "-q", "--no-header", "-p", "no:cacheprovider", "-p", "tests.conftest",
                        "--rootdir", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=1500)
    tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-2000:]
    assert r.returncode == 0, r.stdout[-6000:]
    assert " passed" in tail and "failed" not in tail and "error" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 90, tail          # the whole module ran (94 cases at the time of writing)


def test_full_forward_gpu_tests_pass_on_emulated_operators(tmp_path):
    """tests/test_gpu_forward.py (golden stage-wise parity in the accurate configuration, mixed batch, zero-match corner,
    product-mode bounds, rectangular pair + batch invariance, 480x640 corner error) with the operators emulated: the HOST
    side of every one of those GPU tests is exercised on CPU.  (The 768x768 / 840x840 shape cases are left to the GPU.)"""
    dst = str(tmp_path / "emulated_test_gpu_forward.py")
    emulated_copy(os.path.join(ROOT, "tests", "test_gpu_forward.py"), dst)
    r = subprocess.run([sys.executable, "-m", "pytest", dst, "-q", "--no-header", "-p", "no:cacheprovider", "-p", "tests.conftest",
                        "--rootdir", str(tmp_path), "-k", "not fire_and_megadepth"], capture_output=True, text=True, cwd=ROOT,
                       timeout=1500)
    tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-2000:]
    assert r.returncode == 0, r.stdout[-6000:]
    assert " passed" in tail and "failed" not in tail and "error" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 8, tail


def test_emulations_pass_the_kernel_tests_at_scale(tmp_path):
    """tests/test_gpu_kernels_at_scale.py with the operators emulated: its own host logic - the premise assertions (lazy
    raises counted, leads in (6, 8], mixed warps, ring wraps, chunk sizes covered), the broken-reference sensitivity checks
    and the fp64 references - runs in the CPU suite.  The batch-16 matcher case (several GB of fp32 confidences on the
    CPU) is left to the GPU."""
    dst = str(tmp_path / "emulated_test_gpu_kernels_at_scale.py")
    emulated_copy(os.path.join(ROOT, "tests", "test_gpu_kernels_at_scale.py"), dst)
    r = subprocess.run([sys.executable, "-m", "pytest", dst, "-q", "--no-header", "-p", "no:cacheprovider", "-p", "tests.conftest",
                        "--rootdir", str(tmp_path), "-k", "not batch16"], capture_output=True, text=True, cwd=ROOT,
                       timeout=1500)
    tail = r.stdout.strip().splitlines()[-1] if r.stdout.strip() else r.stderr[-2000:]
    assert r.returncode == 0, r.stdout[-6000:]
    assert " passed" in tail and "failed" not in tail and "error" not in tail, tail
    assert int(tail.split(" passed")[0].split()[-1]) >= 17, tail


def test_smoke_entry_point_on_emulated_operators(monkeypatch, capsys):
    """__graft_entry__.smoke() (the driver's round-end check on cuda:0: shipped configuration vs the oracle) with the
    operators emulated: its own logic and thresholds hold when the arithmetic behind the contracts is exact."""
    import torch
    from geoformer_b200 import _lib
    from geoformer_b200.model.full_model import GeoFormer
    from tests import emu_ops
    emu_ops.install(monkeypatch)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(GeoFormer, "forward", lambda self, data: self._forward(data, data["image0"], data["image1"]))
    monkeypatch.setattr(_lib, "launch_count", lambda: sum(emu_ops.CALLS.values()))
    src = open(os.path.join(ROOT, "__graft_entry__.py")).read()
    assert src.count('"cuda:0"') == 1 and src.count(".cuda()") == 2
    src = src.replace('"cuda:0"', '"cpu"').replace(".cuda()", ".cpu()")
    g = {"__name__": "graft_entry_emulated", "__file__": os.path.join(ROOT, "__graft_entry__.py")}
    exec(compile(src, "__graft_entry__.py", "exec"), g)
    g["smoke"]()
    out = capsys.readouterr().out
    assert "smoke (product mode)" in out and "overlap" in out
