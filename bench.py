#!/usr/bin/env python
"""Benchmark of the GeoFormer matching hot path (BASELINE.json metric: 640x480 pairs/s on B200;
conf-matrix tensor-pipe fraction of peak).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the full forward (backbone -> coarse transformer -> coarse matching ->
host RANSAC -> geo transformer -> coarse matching -> fine stage) over one batch of synthetic
HPatches-shaped 640x480 pairs.  Prints ONE JSON line on rank 0.  Inputs and weights are seeded, so
the outputs written by --dump-outputs can be compared between two builds of the project.
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from geoformer_b200 import synth  # noqa: E402

H, W, BATCH = 480, 640, 16
METRIC, UNIT = "pairs_per_sec_640x480", "pairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--regime", default="dense", choices=["dense", "shift"])
    ap.add_argument("--backbone", default=os.environ.get("GF_BACKBONE", "f16"))
    ap.add_argument("--ransac", default=os.environ.get("GF_RANSAC", "cv2"), choices=["cv2", "gpu"],
                    help="cv2 = host cv2.findHomography as the reference (default); gpu = csrc/ransac.cu (not bit-identical)")
    ap.add_argument("--depth", type=int, default=3, help="batches in flight (MatchPipeline); 1 = plain serial forward")
    ap.add_argument("--hw", default=None, help="HxW override for informational runs of the other BASELINE configs (e.g. 768x768)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stage-times", action="store_true", help="print a per-stage CUDA-event breakdown to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output arrays of the last timed step as DIR/<name>.npy "
                         "(rank 0 only; float32, or float64 for float64 and integer outputs; at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def workload_config(args, extra=None):
    shape = {(480, 640): "HPatches-shaped synthetic 640x480", (768, 768): "FIRE-shaped synthetic 768x768 (9216 coarse tokens)",
             (840, 840): "MegaDepth-shaped synthetic 840x840 (11025 coarse tokens, high match count)"}.get((H, W), f"synthetic {W}x{H}")
    cfg = {"workload": f"{shape} pairs, batch {args.batch}, regime '{args.regime}' "
                       f"(image1 == image0: heaviest match count), random-init weights, coarse_thr 0.0",
           "image_hw": [H, W], "pairs_per_step": args.batch, "coarse_tokens": (H // 8) * (W // 8),
           "cache": "working set per step (activations > 3 GB per batch, several batches in flight) >> 126 MB L2; no explicit flush"}
    if extra:
        cfg.update(extra)
    return cfg


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, out_dir, limit=DUMP_LIMIT_BYTES):
    """Write every tensor of one step's output dict as <out_dir>/<name>.npy: floating tensors as float32 (float64 stays
    float64), integer and bool tensors as float64, which holds them exactly.  Above `limit` bytes in all, arrays of more
    than one row keep a fixed, seeded sample of their rows (arrays of the same length keep the same rows), so that two
    runs stay comparable row for row."""
    arrs = {}
    for k, v in outputs.items():
        if not torch.is_tensor(v):
            continue
        a = v.detach().cpu().numpy()
        arrs[k] = a.astype(np.float32 if np.issubdtype(a.dtype, np.floating) and a.dtype != np.float64 else np.float64)
    big = [k for k, a in arrs.items() if a.ndim and a.shape[0] > 1]
    rest = sum(a.nbytes for k, a in arrs.items() if k not in big)
    total = rest + sum(arrs[k].nbytes for k in big)
    if total > limit:
        keep = (limit - rest) / (total - rest)
        for k in big:
            a = arrs[k]
            rows = np.random.default_rng(0).choice(a.shape[0], max(1, int(a.shape[0] * keep)), replace=False)
            arrs[k] = a[np.sort(rows)]
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a)


# ------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock / throttle-reason samples under the bench load, through NVML in-process (nvidia_ml_py).
    Every query goes through the driver's GPU lock and, about once in a hundred calls, stalled the kernel-launching
    threads for ~100 ms (a looping `nvidia-smi` subprocess was worse): with 100 ms polling one timed loop in six lost a
    whole step to it, without any polling none in 15 runs did.  So the timed loops are sampled sparsely (every 300 ms,
    2-3 samples each) and the same load is run once more, untimed, with dense sampling; all samples are reported."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.samples, self.first, self.stop_flag, self.thread, self.h = index, [], 0, False, None, None
        self.interval, self.timed_samples = 0.3, 0

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.h = None

    def _pump(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((mhz, mask))
            except Exception:
                pass
            time.sleep(self.interval)

    def mark(self):
        """Samples from here on belong to the timed region."""
        self.first = len(self.samples)

    def stop(self):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        use = self.samples[self.first:] or self.samples
        reasons = sorted({nm for _, mask in use for nm, bit in self.REASONS if mask & bit})
        return {"sm_mhz": float(np.median([m for m, _ in use])) if use else None, "sm_max_mhz": self.max_mhz,
                "samples": len(use), "samples_inside_timed_loops": self.timed_samples, "reasons": reasons}


# ------------------------------------------------------------------------------------------- reference arm / CPU baseline
def cpu_forward_pairs_per_sec(steps, warmup, regime):
    """The reference's CPU implementation of the path == the oracle port (the reference is pure PyTorch and cannot
    travel to the GPU box; the oracle restates it op for op and is pinned to it by tests/golden).  Each step is a
    bounded sample of the workload: ONE 640x480 pair (about 5 s of CPU work)."""
    from oracle import geoformer_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth.make_state_dict(0)
    times = []
    for i in range(warmup + steps):
        im0, im1 = synth.make_pairs(1, H, W, regime, 100 + i)
        t0 = time.perf_counter()
        with torch.no_grad():
            out = O.forward(sd, im0, im1, dict(coarse_thr=0.0))
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return 1.0 / float(np.mean(times)), torch.get_num_threads(), float(np.mean(times)), out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    v, cores, spp, out = cpu_forward_pairs_per_sec(steps, warmup, args.regime)
    if args.dump_outputs:
        dump_outputs(out, args.dump_outputs)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": 1e3 * spp, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, {"pairs_per_step": 1,
                                             "steps_note": "CPU arm: each step is ONE pair (~2-5 s of all-core CPU work)"}),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{steps} single-pair {W}x{H} forwards of the CPU oracle port after {warmup} warm-up "
                                       f"(the reference is pure PyTorch; the oracle restates it op for op)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


# ------------------------------------------------------------------------------------------- our arm
def build_model(device, backbone, ransac="cv2"):
    from geoformer_b200.model.full_model import GeoFormer
    from geoformer_b200.model.geo_config import default_cfg as geo_cfg
    from geoformer_b200.model.loftr_src.loftr.utils.cvpr_ds_config import default_cfg
    g = dict(geo_cfg)
    g["coarse_thr"] = 0.0
    m = GeoFormer(copy.deepcopy(default_cfg), g)
    ckpt = {"state_dict": {"matcher." + k: v for k, v in synth.make_state_dict(0).items()}}   # checkpoint-shaped, as the wrapper loads it
    m.load_state_dict(ckpt["state_dict"], strict=False)
    m.backbone_precision = backbone
    m.ransac = ransac
    return m.eval().to(device)


def run_ours(args):
    import torch.distributed as dist
    from geoformer_b200 import _lib, ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import datetime
        # a collective mismatch between ranks must fail within minutes, not after NCCL's default 10-minute watchdog
        dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=180))
    model = build_model(device, args.backbone, args.ransac)

    # a small pool of distinct batches, resident in HBM (value) and in pinned host memory (e2e)
    pool = 2
    host = [synth.make_pairs(args.batch, H, W, args.regime, 1000 * rank + 100 * p) for p in range(pool)]
    host = [(a.pin_memory(), b.pin_memory()) for a, b in host]
    dev = [(a.to(device), b.to(device)) for a, b in host]

    from geoformer_b200.pipeline import MatchPipeline
    pipe = MatchPipeline(model, depth=args.depth, device=device, freeze_gc=True)

    from geoformer_b200.dist import all_gather_match_block, pack_match_list, reduce_sums, unpack_match_lists
    done_t = []                    # host completion time of every batch (GF_BENCH_TRACE=1 prints the gaps to stderr)
    cap = args.batch * (H // 8) * (W // 8)          # matches per batch <= pairs * L (at most one per coarse row)
    xstream = torch.cuda.Stream(device=device)      # the path's only collective runs here, beside the next batches' compute
    xev = []                                        # CUDA events around every exchange (reported, not part of the timing)
    last_gather = {}
    last_outputs = {}                               # --dump-outputs: the output tensors of the latest batch, in batch order

    def block_of(d):               # packed match list of the batch (device, fixed capacity, no host sync); pair id = global
        return pack_match_list(d["mkpts0_f"], d["mkpts1_f"], d["mconf"], d["m_bids"] * world + rank, cap)

    def counts_only(d):            # keep only what the report needs (frees the big per-batch tensors early)
        done_t.append(time.perf_counter())
        res = {"b_ids": d["b_ids"].shape[0], "mkpts0_f": d["mkpts0_f"].shape[0], "block": block_of(d)}
        if args.dump_outputs:      # references only: no copy and no sync inside the timed loop
            res["outputs"] = {k: v for k, v in d.items() if k not in ("image0", "image1")}
        return res

    def to_host(d):                # what match_pairs() reads back (geoformer.py:53-54,73)
        k0, k1, cf = d["mkpts0_f"].cpu(), d["mkpts1_f"].cpu(), d["mconf"].cpu()
        return counts_only(d), k0.numel() * 4 + k1.numel() * 4 + cf.numel() * 4

    def exchange(block):
        """Gather this batch's match list over all ranks: ONE all_gather_into_tensor of the packed int32 block, issued
        from the main thread in batch order (same order on every rank) on a side stream."""
        block.record_stream(xstream)       # allocated on a worker's stream, consumed here
        with torch.cuda.stream(xstream):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out, _ = all_gather_match_block(block)
            e1.record()
        xev.append((e0, e1))
        last_gather["blocks"] = out

    def drive(batches, post, collective=True):
        """collective=False: a pass that only SOME ranks run (rank 0's densely clock-sampled repeat) must not issue the
        all-gather - every rank has to execute the same sequence of collectives (an r02 8-GPU attempt hung on exactly
        this: rank 0 issued extra all-gathers while the others waited in the final all-reduce)."""
        outs = []
        for res in pipe.run_iter(batches, post):
            r = res[0] if isinstance(res, tuple) else res
            blk = r.pop("block")
            last_outputs["outputs"] = r.pop("outputs", None)
            if collective:
                exchange(blk)
            outs.append(res)
        return outs

    def run_resident(steps, collective=True):
        return drive(({"image0": dev[i % pool][0], "image1": dev[i % pool][1]} for i in range(steps)), counts_only, collective)

    def run_e2e(steps):
        return drive(({"image0": host[i % pool][0], "image1": host[i % pool][1]} for i in range(steps)), to_host)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record()
        outs = fn(steps)
        torch.cuda.current_stream().wait_stream(xstream)      # the exchanges belong to the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, outs, _lib.launch_count() - l0

    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("GF_BENCH_NO_CLOCKS"):
        sampler.start()
    run_resident(args.warmup)
    run_e2e(args.warmup)
    # Settle pass (untimed, on top of the W warm-up steps): ~1.5 s of the same load.  The board reaches its power cap
    # about a second into sustained load; the clock step-down that follows cost one timed loop in three a 100-300 ms
    # stall when it fell inside it (0 of 7 runs with the settle pass, also 0 of 15 without NVML polling).
    settle = max(args.warmup, int(os.environ.get('GF_BENCH_PREWARM', '40')))
    run_resident(settle)
    sampler.mark()
    done_t.clear()
    ms, outs, launches = timed(run_resident, args.steps)
    step_outputs = last_outputs.pop("outputs", None)
    if os.environ.get("GF_BENCH_TRACE") and rank == 0:
        print("value loop, ms between batch completions:", " ".join(f"{1e3 * (b - a):.0f}" for a, b in zip(done_t, done_t[1:])),
              file=sys.stderr)
    ms_e2e, outs_e2e, _ = timed(run_e2e, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(step_outputs, args.dump_outputs)
    if rank == 0 and sampler.h is not None:      # same load once more, untimed, densely sampled (see ClockSampler)
        sampler.timed_samples = len(sampler.samples) - sampler.first
        sampler.interval = 0.04
        run_resident(max(4, args.steps // 2), collective=False)      # rank 0 only: no collective in here
        sampler.interval = 0.3
    # dominant-kernel timing, live in this run: the two tcgen05 passes of the conf-matrix kernel (statistics pass and
    # confidence pass; each launch contracts the full n x L x S x C problem), CUDA events on the launching stream
    L_ = (H // 8) * (W // 8)
    g = torch.Generator(device=device).manual_seed(1)
    fa = torch.randn(args.batch, L_, 256, device=device, generator=g) * 3 + 1.5
    fb = torch.randn(args.batch, L_, 256, device=device, generator=g) * 3 + 1.5
    a3 = torch.empty((args.batch, L_, 768), device=device, dtype=torch.float16); b3 = torch.empty_like(a3)
    st = torch.cuda.current_stream().cuda_stream
    _lib.call("gf_pack_split_f16", fa.data_ptr(), a3.data_ptr(), args.batch * L_, 256, 1 / 16, 0, st)
    _lib.call("gf_pack_split_f16", fb.data_ptr(), b3.data_ptr(), args.batch * L_, 256, 1 / 16, 1, st)
    ws = torch.empty(_lib.load().gf_coarse_match_fused_workspace_bytes(args.batch, L_, L_), device=device, dtype=torch.uint8)
    mj = torch.empty(args.batch * L_, device=device, dtype=torch.int32); mcf = torch.empty(args.batch * L_, device=device)
    _lib.call("gf_coarse_match_fused", a3.data_ptr(), b3.data_ptr(), args.batch, L_, L_, 768, 10.0, 0.0, 0, H // 8, W // 8,
              H // 8, W // 8, ws.data_ptr(), mj.data_ptr(), mcf.data_ptr(), st)
    sim_ms = []
    for it in range(6):
        for ps in (0, 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.call("gf_coarse_match_fused_pass", a3.data_ptr(), b3.data_ptr(), args.batch, L_, L_, 768, 10.0,
                      ws.data_ptr(), ps, st)
            e1.record()
            if it >= 2:
                sim_ms.append((e0, e1))
    torch.cuda.synchronize()
    sim_ms = [a.elapsed_time(b) for a, b in sim_ms]
    del fa, fb, a3, b3, ws
    # the largest single kernel of a step by time: one fused fine-level layer over both images' windows (self layer)
    fl_ms, fl_windows = [], 0
    try:
        wp = model._weights(device).fine[0]
        fl_windows = 2 * int(round(float(np.mean([o["b_ids"] for o in outs]))))
        if fl_windows > 0 and "wpack" in wp:
            xf = torch.randn(fl_windows, 25, 128, device=device)
            yf = torch.empty_like(xf)
            for it in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _lib.call("gf_fine_layer", xf.data_ptr(), xf.data_ptr(), wp["wpack"].data_ptr(), wp["n1w"].data_ptr(),
                          wp["n1b"].data_ptr(), wp["n2w"].data_ptr(), wp["n2b"].data_ptr(), yf.data_ptr(), fl_windows, st)
                e1.record()
                if it >= 2:
                    fl_ms.append((e0, e1))
            torch.cuda.synchronize()
            fl_ms = [a.elapsed_time(b) for a, b in fl_ms]
            del xf, yf
    except Exception:
        fl_ms = []
    # projection GEMMs of one coarse-transformer layer in their shipped variants, timed live (rows = both images of the batch)
    gemm_ms = []
    try:
        from geoformer_b200.ops import EPI_ELU1, EPI_LN, EPI_RELU
        lw = model._weights(device).coarse[0]
        m_rows = 2 * args.batch * L_
        gx = torch.randn(m_rows, 256, device=device)
        q_ = ops.linear(gx, lw["wqkv"], epi=EPI_ELU1, act_cols=512, out_f16=True)
        msg_ = q_[:, :256].contiguous()
        n1_ = ops.linear(msg_, lw["wm16"], epi=EPI_LN, gamma=lw["n1w"], beta=lw["n1b"])
        h_ = ops.linear(gx, lw["w1"], a2=n1_, epi=EPI_RELU, out_f16=True)
        calls = [lambda: ops.linear(gx, lw["wqkv"], epi=EPI_ELU1, act_cols=512, out_f16=True),
                 lambda: ops.linear(msg_, lw["wm16"], epi=EPI_LN, gamma=lw["n1w"], beta=lw["n1b"]),
                 lambda: ops.linear(gx, lw["w1"], a2=n1_, epi=EPI_RELU, out_f16=True),
                 lambda: ops.linear(h_, lw["w2_16"], epi=EPI_LN, gamma=lw["n2w"], beta=lw["n2b"], residual=gx)]
        for fn in calls:
            evs = []
            for it in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record()
                if it >= 2:
                    evs.append((e0, e1))
            torch.cuda.synchronize()
            gemm_ms.append(float(np.mean([a.elapsed_time(b) for a, b in evs])))
        del gx, q_, msg_, n1_, h_
    except Exception as e:      # diagnostic block only
        print("gemm timing skipped:", e, file=sys.stderr)
        gemm_ms = []
    clocks = sampler.stop() if rank == 0 else None

    mc = float(np.mean([o["b_ids"] for o in outs])) / args.batch
    mf = float(np.mean([o["mkpts0_f"] for o in outs])) / args.batch
    d2h = int(np.mean([o[1] for o in outs_e2e]))
    # the path's only exchange step ran inside the timed loops (one all_gather_into_tensor per batch); its device time:
    torch.cuda.synchronize()
    xms = [a.elapsed_time(b) for a, b in xev[-2 * args.steps:]]
    exchange_ms = float(np.mean(xms)) if xms else 0.0
    allm, allid = unpack_match_lists(last_gather["blocks"])
    gathered = int(allm.shape[0])
    mc, mf = [v / world for v in reduce_sums([mc, mf], device)]
    try:
        other = other_configs(args, rank, world, device, drive)
    except Exception as e:          # noqa: BLE001 - informational block (even a failed collective in it must not cost the line)
        other = {"failed": True, "error": f"{type(e).__name__}: {e}"[:200]}
    if args.stage_times and rank == 0:
        stage_breakdown(model, dev[0])
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pairs = args.batch * args.steps * world
    value = pairs / (ms / 1e3)
    e2e = pairs / (ms_e2e / 1e3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained"
    # ncu evidence committed under profiles/ (tools/ncu_summary.py of `ncu --set full` on tools/prof_r02_ncu.py, same shapes)
    ncu = {}
    try:
        for k in json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_main_kernels.json")))["kernels"]:
            ncu.setdefault(k["kernel"], []).append(k)
    except Exception:
        pass

    def ncu_of(name, idx=0):
        v = ncu.get(name)
        return v[min(idx, len(v) - 1)] if v else None

    L = (H // 8) * (W // 8)
    flops = 2.0 * L * L * 256 * args.batch                                   # algorithmic: 2*L*S*C per pair per launch
    sim_avg_ms = float(np.mean(sim_ms)) if len(sim_ms) else float("nan")
    achieved = flops / (sim_avg_ms * 1e-3) / 1e12
    n0, n1 = ncu_of("sim_fused_kernel<0>"), ncu_of("sim_fused_kernel<1>")
    roof = {"kernel": "sim_fused_kernel<pass 0|1> (coarse similarity contraction on CTA pairs, split-fp16 K=768, dual-softmax "
                      "fused into the epilogue; average over the two passes)",
            "bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
            "peak_source": peak_src,
            "algorithmic_flops_per_launch": flops, "issued_flops_per_launch": 3 * flops,
            "issued_frac": 3 * achieved / peak_tf,      # tensor-pipe view: the split-fp16 product issues 3 MMAs per algorithmic one
            "avg_launch_ms": sim_avg_ms, "launches_timed": len(sim_ms),
            # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture (16 pairs), scaled to this
            # batch; algorithmic bytes per launch = packed operands 235.9 MB (+ 105 MB statistics partials in pass 0)
            "traffic": (0.5 * (n0["dram_bytes"] + n1["dram_bytes"]) * args.batch / 16) if n0 and n1 else None,
            "traffic_source": "profiles/r02_ncu_main_kernels.json" if n0 else None,
            "tensor_pipe_active_pct_ncu": {"pass0": n0["tensor_pipe_pct"], "pass1": n1["tensor_pipe_pct"],
                                           "sm_clock_ghz_under_ncu": [n0["sm_clock_ghz"], n1["sm_clock_ghz"]]} if n0 and n1 else None}
    roof2 = None
    if fl_ms:
        fl_avg = float(np.mean(fl_ms))
        # algorithmic FLOPs of one fine-level layer application: per 25-token window q/k/v/merge 4 x 2*25*128*128, MLP
        # 2*25*256*256 + 2*25*256*128, linear attention ~0.2 M  =  8.4 MFLOP (SURVEY 8d: 33.6 MFLOP per match / 4 applications)
        fl_flops = fl_windows * 8.4e6
        nf = ncu_of("fl::fine_layer_kernel")
        roof2 = {"kernel": "fine_layer_kernel (one whole fine-level LoFTR layer per launch, self layer over both images' "
                           "windows; qkv / attention / merge / LN / MLP / LN / residual never leave the SM)",
                 "bound": "tensor", "achieved": fl_flops / (fl_avg * 1e-3) / 1e12, "peak": peak_tf, "unit": "TFLOP/s",
                 "frac": fl_flops / (fl_avg * 1e-3) / 1e12 / peak_tf, "peak_source": peak_src,
                 "algorithmic_flops_per_launch": fl_flops, "windows": fl_windows, "avg_launch_ms": fl_avg,
                 "algorithmic_bytes_per_launch": fl_windows * 25 * 128 * 4 * 2.0,      # x read once + y written once (HBM view)
                 "traffic": (nf["dram_bytes"] * fl_windows / 130898.0) if nf else None,
                 "traffic_source": "profiles/r02_ncu_main_kernels.json (130898 windows), scaled" if nf else None,
                 "tensor_pipe_active_pct_ncu": nf["tensor_pipe_pct"] if nf else None}
    line_gemms = None
    if gemm_ms:
        m_rows = 2 * args.batch * L
        spec = {"qkv 768x256 (tf32 in, fp16 out, elu+1)": (2.0 * m_rows * 768 * 256, m_rows * (256 * 4 + 768 * 2), "gemm_tc_kernel<0, 256, 0, 1, 1>"),
                "merge 256x256 (fp16 in, LayerNorm)": (2.0 * m_rows * 256 * 256, m_rows * (256 * 2 + 256 * 4), "gemm_tc_kernel<1, 256, 1, 1, 0>"),
                "mlp.0 512x512 (tf32 in, fp16 out, ReLU)": (2.0 * m_rows * 512 * 512, m_rows * (512 * 4 + 512 * 2), "gemm_tc_kernel<0, 256, 0, 1, 1>"),
                "mlp.2 256x512 (fp16 in, LayerNorm + residual)": (2.0 * m_rows * 512 * 256, m_rows * (512 * 2 + 256 * 4 + 256 * 4), "gemm_tc_kernel<1, 256, 1, 1, 0>")}
        hbm = float(peaks.get("hbm_gbs", 6500.0))
        line_gemms = {}
        for (name, (fl_, by_, kn)), t_ms in zip(spec.items(), gemm_ms):
            nk = ncu_of(kn, 1 if name.startswith("mlp.2") else 0)
            line_gemms[name] = {"avg_launch_ms": t_ms, "tflops": fl_ / (t_ms * 1e-3) / 1e12, "frac_of_tensor_peak": fl_ / (t_ms * 1e-3) / 1e12 / peak_tf,
                                "hbm_gbs_algorithmic": by_ / (t_ms * 1e-3) / 1e9, "frac_of_hbm_peak": by_ / (t_ms * 1e-3) / 1e9 / hbm,
                                "bound": "hbm" if by_ / hbm / 1e9 > fl_ / peak_tf / 1e12 else "tensor",
                                "tensor_pipe_active_pct_ncu": nk["tensor_pipe_pct"] if nk else None,
                                "dram_pct_ncu": nk["dram_pct"] if nk else None}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": ("tf32 / fp16 tensor-core operands with fp32 accumulation (fp32 residual stream, fp16 intermediates), "
                      f"split-fp16 similarity, {args.backbone} backbone activations"),
            "data": "synthetic",
            "config": workload_config(args, {"matches_coarse_per_pair": mc, "matches_fine_per_pair": mf,
                                             "batches_in_flight": args.depth, "ransac": args.ransac,
                                             "untimed_steps_before_timing": f"{args.warmup} warm-up (resident) + {args.warmup} warm-up (host inputs) + {settle} power-cap settle", "exchange": "inside the timed region: one all_gather_into_tensor per batch (int16 coordinates + fp32 confidence + pair id, 16 B per match, fixed capacity, no host sync) on a side stream",
                                             "exchange_ms_per_batch": exchange_ms, "exchange_bytes_per_rank_per_batch": (cap + 1) * 16,
                                             "gathered_matches_last_batch_all_ranks": gathered,
                                             "parallelism": f"pairs sharded over {world} GPU(s), no data-path collective",
                                             "other_baseline_configs": other}),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": 2 * args.batch * H * W * 4, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_top_kernel_by_time": roof2,
            "roofline_projection_gemms": line_gemms}
    if not args.no_cpu_baseline and world == 1:
        v, cores, spp, _ = cpu_forward_pairs_per_sec(2, 1, args.regime)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"2 single-pair {W}x{H} forwards of the CPU oracle port after 1 warm-up "
                                          f"({spp:.2f} s/pair)"}
    else:
        line["cpu_baseline"] = None
    _emit(line)
    if world > 1:
        dist.destroy_process_group()


def other_configs(args, rank, world, device, drive, steps=4, warmup=2):
    """BASELINE.json configs[3] / configs[4] — FIRE-shaped 768x768 and MegaDepth-shaped 840x840 pairs — measured in the
    same run on the same N GPUs as an INFORMATIONAL block of the line (the headline metric stays the 640x480 one): same
    batch size, regime, weights and pipeline depth; inputs resident in HBM, `steps` timed steps after `warmup`, CUDA
    events, max over ranks; no match-list exchange here.  GF_BENCH_EXTRA_HW overrides the shape list ("" disables).
    Every collective below is issued unconditionally by every rank (a rank whose measurement failed contributes a
    failure flag), so a failure cannot desynchronise the ranks."""
    import torch.distributed as dist
    from geoformer_b200.dist import reduce_sums
    if (H, W) != (480, 640) and "GF_BENCH_EXTRA_HW" not in os.environ:      # only beside the headline workload, not on --hw runs
        return None
    out = {}
    post = lambda d: {"b_ids": d["b_ids"].shape[0], "mkpts0_f": d["mkpts0_f"].shape[0], "block": None}
    for spec in [x for x in os.environ.get("GF_BENCH_EXTRA_HW", "768x768,840x840").split(",") if x.strip()]:
        ms, failed, mcx, mfx, err = -1.0, 0.0, 0.0, 0.0, None
        try:
            eh, ew = (int(v) for v in spec.lower().split("x"))
            xin = [tuple(t.to(device) for t in synth.make_pairs(args.batch, eh, ew, args.regime, 7000 + 1000 * rank + 100 * p))
                   for p in range(2)]
            gen = lambda k: ({"image0": xin[i % 2][0], "image1": xin[i % 2][1]} for i in range(k))
            drive(gen(warmup), post, False)                       # allocator blocks and position tables of this shape
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = drive(gen(steps), post, False)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            mcx = float(np.mean([r["b_ids"] for r in res])) / args.batch
            mfx = float(np.mean([r["mkpts0_f"] for r in res])) / args.batch
            del xin, res
        except Exception as e:                  # noqa: BLE001 - informational block: never costs the headline line
            failed, err = 1.0, f"{type(e).__name__}: {e}"[:200]
            print(f"other config {spec} failed on rank {rank}: {err}", file=sys.stderr)
        t = torch.tensor([ms, failed], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mcx, mfx = [v / world for v in reduce_sums([mcx, mfx], device)]
        ms_max, any_failed = float(t[0].item()), bool(t[1].item() > 0)
        out[spec] = ({"failed": True, "error_rank0": err} if any_failed or ms_max <= 0 else
                     {"pairs_per_sec": args.batch * steps * world / (ms_max / 1e3), "ms_per_step": ms_max / steps, "steps": steps,
                      "warmup": warmup, "pairs_per_step": args.batch, "coarse_tokens": (eh // 8) * (ew // 8),
                      "matches_coarse_per_pair": mcx, "matches_fine_per_pair": mfx,
                      "note": "informational: resident inputs, CUDA events, max over ranks, no exchange"})
    return out


def stage_breakdown(model, batch):
    """Per-stage CUDA-event timing (diagnostic; stderr)."""
    from geoformer_b200 import ops
    ops.PROFILE.enable("*")
    model({"image0": batch[0], "image1": batch[1]})
    torch.cuda.synchronize()
    rows = ops.PROFILE.summary()
    ops.PROFILE.disable()
    tot = sum(v[1] for k, v in rows.items() if k.startswith("stage:"))
    for k, (cnt, ms) in sorted(rows.items(), key=lambda kv: (not kv[0].startswith("stage:"), -kv[1][1])):
        sys.stderr.write(f"  {k:36s} x{cnt:4d}  {ms:9.3f} ms  {100 * ms / tot:5.1f}%\n")
    sys.stderr.write(f"  {'sum of stages':36s}        {tot:9.3f} ms\n")


def _emit(line: dict) -> None:
    """Exactly ONE JSON line on the real stdout (fd 1 was pointed at stderr while the run was in progress so that
    library chatter such as NCCL's version banner cannot pollute it)."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)

if __name__ == "__main__":
    a = parse()
    if a.hw:
        H, W = [int(v) for v in a.hw.lower().split("x")]
        METRIC = f"pairs_per_sec_{W}x{H}"
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
