"""Host-side logic that needs no GPU: the ordered-iterator pipeline (results in input order, error propagation) and the
reference arm of bench.py (contract keys of its JSON line)."""
import json
import os
import random
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _StubPipeline:
    """MatchPipeline with the CUDA plumbing stubbed out: exercises the worker / ordering / error logic of run_iter."""

    def __new__(cls, depth, fail_at=None, monkeypatch=None):
        from geoformer_b200.pipeline import MatchPipeline

        class Stream:
            def wait_stream(self, s):
                pass

        class Dev:
            def __init__(self, *a):
                pass

            def __enter__(self):
                return self

            def __exit__(self, *a):
                return False

        monkeypatch.setattr(torch.cuda, "current_stream", lambda d=None: Stream())
        monkeypatch.setattr(torch.cuda, "device", Dev)
        monkeypatch.setattr(torch.cuda, "set_device", lambda d: None)

        class P(MatchPipeline):
            def __init__(self):
                self.depth, self.streams, self.freeze_gc, self._frozen, self.device = depth, [], False, False, None
                self.model = type("M", (), {"_weights": lambda self, d: None})()

            def _job(self, slot, data, post):
                time.sleep(random.random() * 0.005)
                if fail_at is not None and data["i"] == fail_at:
                    raise RuntimeError("boom")
                return data["i"] if post is None else post(data)

        return P()


@pytest.mark.parametrize("depth", [1, 2, 4])
def test_run_iter_yields_in_input_order(depth, monkeypatch):
    p = _StubPipeline(depth, monkeypatch=monkeypatch)
    seen = []
    for r in p.run_iter(({"i": i} for i in range(41))):
        seen.append(r)                       # the consumer runs on the calling thread, in batch order
    assert seen == list(range(41))
    assert p.run([]) == []
    assert p.run(({"i": i} for i in range(5)), post=lambda d: d["i"] * 2) == [0, 2, 4, 6, 8]


def test_run_iter_propagates_worker_errors(monkeypatch):
    p = _StubPipeline(3, fail_at=7, monkeypatch=monkeypatch)
    got = []
    with pytest.raises(RuntimeError, match="boom"):
        for r in p.run_iter(({"i": i} for i in range(30))):
            got.append(r)
    assert got == list(range(len(got))) and len(got) <= 7       # everything before the failing batch, in order


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the oracle port timed on the host cores): one JSON line on stdout with the contract's
    keys; under torchrun only rank 0 prints."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--hw", "96x128"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "steps_note" in d["config"] and d["steps"] == 1 and d["warmup"] == 0
    # a non-zero rank prints nothing and exits 0
    r2 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                        capture_output=True, text=True, timeout=120, env=dict(os.environ, RANK="1", WORLD_SIZE="2"), cwd=ROOT)
    assert r2.returncode == 0 and r2.stdout.strip() == ""


def _dryrun(world, extra_env=None, timeout=420, extra_args=()):
    """bench.py's own arm on `world` simulated ranks (tests/bench_dryrun.py: operators emulated on CPU, gloo for NCCL)."""
    import socket
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), LOCAL_RANK=str(r), WORLD_SIZE=str(world), LOCAL_WORLD_SIZE=str(world),
                   MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), OMP_NUM_THREADS="2", GF_BENCH_EXTRA_HW="64x64,72x88",
                   **(extra_env or {}))
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, "tests", "bench_dryrun.py"), "--gpus", str(world), "--steps", "3",
                                       "--warmup", "1", "--batch", "2", "--hw", "64x96", "--no-cpu-baseline", "--depth", "2",
                                       *extra_args],
                                      stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env, cwd=ROOT))
    outs = []
    deadline = time.time() + timeout
    for p in procs:
        try:
            o, e = p.communicate(timeout=max(1, deadline - time.time()))
        except subprocess.TimeoutExpired:
            for q in procs:
                q.kill()
            return None
        outs.append((p.returncode, o, e))
    return outs


@pytest.mark.parametrize("world", [1, 2])
def test_bench_own_arm_control_flow_dry_run(world, tmp_path):
    """The whole of bench.py's own arm — warm-up, settle, both timed loops through MatchPipeline, the per-batch
    match-list exchange, barriers, max-over-ranks, the rank-0-only densely sampled pass, the diagnostics blocks and the
    JSON line — runs to completion on every simulated rank, rank 0 prints exactly one line with the contract's keys, the
    other ranks print nothing.  (A collective issued by some ranks only would hang here as it would under NCCL.)
    --dump-outputs: rank 0 writes the output arrays of its last timed batch."""
    dump = tmp_path / "outputs"
    outs = _dryrun(world, extra_args=("--dump-outputs", str(dump)))
    assert outs is not None, "bench.py dry run timed out: the ranks' collective sequences differ"
    for rc, _, err in outs:
        assert rc == 0, err[-3000:]
    lines = [l for l in outs[0][1].splitlines() if l.strip()]
    assert len(lines) == 1 and all(o.strip() == "" for _, o, _ in outs[1:])
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline", "cpu_baseline"):
        assert k in d, k
    assert d["n_gpus"] == world and d["steps"] == 3 and d["scaling"] == "weak" and d["unit"] == "pairs/s"
    assert d["value"] == pytest.approx(2 * 3 * world / (d["ms_per_step"] * 3 / 1e3))              # whole-job pairs / max-over-ranks time
    assert d["e2e"]["h2d_bytes_per_step"] == 2 * 2 * 64 * 96 * 4 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and d["roofline"]["bound"] == "tensor"
    assert d["clocks"]["samples_inside_timed_loops"] >= 0 and d["clocks"]["sm_max_mhz"] == 1965.0   # rank 0 took the sampling branches
    # informational block for BASELINE configs[3] / configs[4] (shapes shrunk for the dry run)
    oc = d["config"]["other_baseline_configs"]
    assert set(oc) == {"64x64", "72x88"} and all(v["pairs_per_sec"] > 0 and v["steps"] == 4 and v["pairs_per_step"] == 2 for v in oc.values())
    assert oc["72x88"]["coarse_tokens"] == 99 and oc["72x88"]["matches_coarse_per_pair"] > 20
    # the exchange gathered the last batch of EVERY rank
    per_rank = d["config"]["matches_fine_per_pair"] * 2
    assert d["config"]["gathered_matches_last_batch_all_ranks"] == pytest.approx(per_rank * world, rel=0.25)
    got = {f.name[:-4]: np.load(f) for f in dump.iterdir()}
    assert {"mkpts0_f", "mkpts1_f", "mconf", "m_bids", "b_ids", "i_ids", "j_ids"} <= set(got)
    assert "image0" not in got and all(a.dtype in (np.float32, np.float64) for a in got.values())
    n = got["mkpts0_f"].shape[0]
    assert n > 0 and got["mkpts0_f"].shape == got["mkpts1_f"].shape == (n, 2) and got["mconf"].shape == got["m_bids"].shape == (n,)
    assert set(np.unique(got["m_bids"])) <= {0.0, 1.0} and got["m_bids"].dtype == np.float64


def test_bench_dump_outputs_dtypes_and_size_limit(tmp_path):
    """bench.dump_outputs: floating tensors as float32 (float64 kept), integers as float64; above the byte limit every
    multi-row array keeps a seeded sample of its rows (the same rows for arrays of the same length), small ones stay whole."""
    code = (f"import sys, torch; sys.path.insert(0, {ROOT!r}); import bench\n"
            "i = torch.arange(20000)\n"
            "out = dict(x=torch.stack([i % 1000, i % 1000 + 1], 1).half(), i=i, d=i.double(), s=torch.tensor(7), t=(1, 2))\n"
            f"bench.dump_outputs(out, {str(tmp_path / 'full')!r})\n"
            f"bench.dump_outputs(out, {str(tmp_path / 'cut')!r}, limit=100000)\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    full = {k: np.load(tmp_path / "full" / f"{k}.npy") for k in ("x", "i", "d", "s")}
    assert not (tmp_path / "full" / "t.npy").exists()
    assert full["x"].dtype == np.float32 and full["i"].dtype == full["d"].dtype == full["s"].dtype == np.float64
    assert np.array_equal(full["x"][:, 1] - 1, np.arange(20000) % 1000) and full["s"] == 7
    cut = {k: np.load(tmp_path / "cut" / f"{k}.npy") for k in ("x", "i", "d", "s")}
    assert sum(a.nbytes for a in cut.values()) <= 100000 and cut["s"] == 7
    assert 0 < cut["i"].shape[0] < 20000 and np.all(np.diff(cut["i"]) > 0)
    assert np.array_equal(cut["i"], cut["d"]) and np.array_equal(cut["x"][:, 0], cut["i"] % 1000)


def test_bench_dry_run_detects_a_rank0_only_collective():
    """Sensitivity check of the dry run: re-injecting the round-2 bug (rank 0's extra pass issuing all-gathers) hangs."""
    assert _dryrun(2, {"GF_DRYRUN_INJECT_RANK0_COLLECTIVE": "1"}, timeout=30) is None


def test_bench_informational_configs_cannot_desynchronise_the_ranks():
    """One rank failing inside the informational 768x768 / 840x840 block (here: rank 1, simulated) neither hangs the run nor
    costs the headline line: every rank still issues the block's collectives, the block reports the failure."""
    outs = _dryrun(2, {"GF_DRYRUN_FAIL_EXTRA_ON_RANK1": "1"})
    assert outs is not None, "hung"
    assert all(rc == 0 for rc, _, _ in outs), outs[1][2][-2000:]
    d = json.loads([l for l in outs[0][1].splitlines() if l.strip()][0])
    assert d["value"] > 0 and d["n_gpus"] == 2
    assert all(v.get("failed") is True for v in d["config"]["other_baseline_configs"].values())
    assert "simulated failure on rank 1" in outs[1][2]
