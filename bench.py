#!/usr/bin/env python
"""Headline benchmark: heads/sec at 256x256 (image -> 413 FLAME params -> 5023x3 vertices -> projected landmarks).

    python bench.py --gpus N --steps K --warmup W                    # this repo (B200-native path), BASELINE configs[1]
    python bench.py --impl reference --gpus N --steps K --warmup W   # the UNMODIFIED reference code on the host CPU cores
    python bench.py --config {2,3,4,5}                               # other BASELINE.json configs (1-based, as SURVEY §8d)

Default workload (config 2 = BASELINE.json configs[1]) per GPU: batch 64 of 256x256 synthetic RGB frames, random-init
weights of the DAD-3DNet architecture, encoder in the fp32-class ``fp16x2`` mode (fp16 hi/lo operands, 22-bit, 3 tensor-core
products, fp32 accumulate; inside the 1e-4 contract, the strict 24-bit ``bf16x3`` mode is timed in the same run under
``strict_fp32_operands``) + FLAME decode + projection + 445-landmark gather.  N>1: every rank runs the same per-GPU batch
on its own shard (weak scaling); constants are broadcast from rank 0 over NCCL at start-up, per-step outputs (params,
vertices, landmarks) are all-gathered on a communication stream that overlaps the next step's encoder.

One JSON line on stdout (rank 0).  ``value`` = whole-job heads/s with inputs resident in HBM; ``e2e`` = the same through
``FaceMeshPredictor.open_stream`` (the public pipelined API) from pinned HOST uint8 frames to pinned HOST results, H2D + D2H
inside the timed region, double-buffered against the compute.  Sub-objects: ``roofline`` (dominant kernel), ``cpu_baseline``,
``decode_microbench`` (config 5), ``config3`` (batch 512, bf16 encoder) at N=1, ``config4`` (512 per GPU) at N>1,
``strict_fp32_operands``, ``parity`` (against the unmodified reference when oracle/_ref is present).

``--dump-outputs DIR`` writes what the timed path returned in its last timed step as ``DIR/<name>.npy`` (float32, or float64
for 64-bit and integer outputs), so that two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "heads/sec @256x256 (5023-vert FLAME)"
UNIT = "heads/s"
FLOPS_PER_IMAGE_ENCODER = 2 * 7_559_801_344        # SURVEY §8(d), analytic
FLOPS_PER_HEAD_BLEND = 13_140_168                  # 2*15069*(400+36), as written in the reference
BYTES_PER_HEAD_DECODE = 413 * 4 + 5023 * 3 * 4     # SURVEY §8(d): params in, vertices out
DUMP_LIMIT_BYTES = 64 << 20

# BASELINE.json `configs`, numbered 1..5 as in SURVEY §8(d)
CONFIGS = {
    1: dict(base="configs[0]: demo.py flame_params on one image through FaceMeshPredictor.__call__", batch=1, precision="fp16x2"),
    2: dict(base="configs[1]: encoder + FLAME decode, fp32-class", batch=64, precision="fp16x2"),
    3: dict(base="configs[2]: full pipeline incl. 445-landmark projection, bf16 encoder / fp32 FLAME", batch=512,
            precision="bf16"),
    4: dict(base="configs[3]: batch 4096 = 8 x 512 sharded across GPUs, NCCL bcast of the FLAME bases + all-gather of vertices",
            batch=512, precision="fp16x2"),
    5: dict(base="configs[4]: FLAME-decode-only microbench, 1M param vectors -> 5023-vertex meshes", batch=1 << 20,
            precision="fp16"),
}

DTYPE = {"fp32": "fp32 operands as bf16x3 split (24-bit), 6 tensor-core products, fp32 accumulate",
         "bf16x3": "fp32 operands as bf16x3 split (24-bit), 6 tensor-core products, fp32 accumulate",
         "fp16x2": "fp32 operands as fp16 hi/lo split (22-bit), 3 tensor-core products, fp32 accumulate (1e-4 contract met; "
                   "strict 24-bit mode timed under strict_fp32_operands)",
         "bf16x2": "bf16 hi/lo split operands (16-bit), fp32 accumulate", "fp16": "fp16 operands, fp32 accumulate",
         "bf16": "bf16 operands, fp32 accumulate"}
PRODUCTS = {"fp32": 6, "bf16x3": 6, "bf16x2": 3, "bf16": 1, "fp16x2": 3, "fp16": 1}


def resolve(args):
    c = CONFIGS[args.config]
    if args.batch is None:
        args.batch = c["batch"]
    if args.precision is None:
        args.precision = c["precision"]
    return args


def workload_config(args, world: int = 1) -> dict:
    """`config` of the JSON line, derived from the arguments actually used (never a hard-coded string)."""
    B = args.batch
    cfg = {"workload": f"{CONFIGS[args.config]['base']} -- batch {B} x 256x256 per GPU, encoder operands {args.precision}, "
                       f"FLAME decode + projection + 445-landmark gather",
           "baseline_config_index": args.config - 1, "per_gpu_batch": B, "global_batch": B * world,
           "encoder_precision": args.precision}
    return cfg


def _traffic_from_profile():
    """DRAM bytes per launch of the dominant kernel, from the committed ncu launch list of this same command
    (profiles/rNN_step_summary_*.json, written by tools/summarize_launches.py).  None when no capture is committed."""
    import glob
    import re

    def ver(f):                                   # r01_step_summary_v11.json -> (1, 11): newest round, newest version
        m = re.search(r"r(\d+)_step_summary_v(\d+)\.json$", f)
        return (int(m.group(1)), int(m.group(2))) if m else (0, 0)
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_step_summary_*.json")), key=ver)
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    return d.get("dominant_dram_bytes_per_launch"), os.path.relpath(files[-1], ROOT)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": d.get("hbm_gbs", 6650.0), "bf16_tflops": d.get("bf16_tflops", 1590.0),
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", 1400.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm = sorted(int(float(s[0])) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit()]
        pw = [float(s[2]) for s in self.samples if s[2].replace(".", "").isdigit()]
        reasons = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, n in enumerate(names):
            if any(s[3 + i].lower().startswith("active") for s in self.samples):
                reasons.append(n)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples), "power_w_max": max(pw) if pw else None}


def dump_outputs(outdir, outputs):
    """Write each output as ``outdir/<name>.npy`` (float32, or float64 for 64-bit and integer outputs).  When they would
    exceed DUMP_LIMIT_BYTES in all, every array keeps the same fraction of its leading-axis rows (heads), drawn with a fixed
    seed, and the kept row indices go to ``outdir/rows_<name>.npy`` (counted in the limit)."""
    import numpy as np
    import torch
    outs = {k: torch.as_tensor(t) for k, t in outputs.items()}
    size = {k: 8 if t.element_size() > 4 or not t.is_floating_point() else 4 for k, t in outs.items()}
    total = sum(t.numel() * size[k] for k, t in outs.items())
    headers = 1024 * (2 * len(outs))                                 # .npy headers, generously
    os.makedirs(outdir, exist_ok=True)
    if total + headers > DUMP_LIMIT_BYTES:
        cost = sum(t.numel() * size[k] + 8 * t.shape[0] for k, t in outs.items())      # data + row index, all rows
        frac = (DUMP_LIMIT_BYTES - headers) / cost
    for k, t in outs.items():
        if total + headers > DUMP_LIMIT_BYTES:
            n = t.shape[0]
            rows = np.sort(np.random.default_rng(0).choice(n, max(1, int(n * frac)), replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
            np.save(os.path.join(outdir, f"rows_{k}.npy"), rows.astype(np.float64))
        a = t.detach().cpu().numpy()
        np.save(os.path.join(outdir, f"{k}.npy"), a.astype(np.float64 if size[k] == 8 else np.float32))


# ------------------------------------------------------------------------------------------------------ reference arm
def _reference_runner(sd):
    """-> (step(x) for a [B,3,256,256] batch, description, kind).  kind "reference": the UNMODIFIED reference code
    (FlameRegression.forward + HeadMesh.vertices_3d + HeadMesh.reprojected_vertices + the 445-index take, i.e. what
    predictor.py:97-142 does per image, batched) through oracle/ref_harness.py -- /root/reference in the build container, its
    byte-compiled twin oracle/_ref on the GPU box; kind "port": the oracle restatement, only when neither exists."""
    import torch
    from oracle import ref_harness as R
    if R.available():
        import warnings
        warnings.filterwarnings("ignore", message="Using torch.cross")
        model = R.flame_regression(sd)
        hm = R.head_mesh()
        from dad_3dheads_b200.flame import load_flame_static
        idx = torch.from_numpy(load_flame_static()["keypoints_445"].astype("int64"))

        def step(x):
            with torch.no_grad():
                res = model(x)                                            # predictor.py:97-100
                p = res["OUTPUT_3DMM_PARAMS"]
                p_out = p.clone()                                         # reprojected_vertices zeroes tz in place (head_mesh.py:41)
                v3 = hm.vertices_3d(p)                                    # predictor.py:136
                pj = hm.reprojected_vertices(params_3dmm=p, to_2d=True)   # predictor.py:137
                return {"3dmm_params": p_out, "points": res["OUTPUT_2D_LANDMARKS"] * 256.0, "3d_vertices": v3,
                        "projected_vertices": pj, "landmarks_445": pj[:, idx]}
        return step, (f"unmodified reference code ({R.kind()} of /root/reference via oracle/ref_harness.py; third-party "
                      "smplx.lbs / pytorchcv ResNet-50 / albumentations from oracle/ref_shims)"), "reference"
    from oracle.predictor_oracle import PredictorOracle
    po = PredictorOracle(sd)
    return po.predict_batch, "oracle restatement (oracle/_ref not built)", "port"


def _best_threads_fn(fn, x_small):
    """torch CPU ops slow down badly when oversubscribed on many-core hosts: time a tiny pass at a few thread counts
    (all cores first) and keep the fastest; the count used is what `cores` reports."""
    import torch
    n = os.cpu_count() or 1
    best, best_t = n, None
    for t in sorted({n, max(1, n // 2), min(n, 32), min(n, 16)}, reverse=True):
        torch.set_num_threads(t)
        fn(x_small)
        t0 = time.perf_counter()
        fn(x_small)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = t, dt
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """The reference's own CPU implementation of the path on the box's host cores: same metric, same config (the full
    per-GPU batch per step), all the host threads it can use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    cfg = workload_config(args, 1)
    B = args.batch
    step, what, kind = _reference_runner(synthetic_state_dict(0))
    x = torch.randn(B, 3, 256, 256, generator=torch.Generator().manual_seed(0))
    cores = _best_threads_fn(step, x[:4])
    for _ in range(args.warmup):
        step(x[:8])                                       # warm-up on a slice: the timed steps below are the full batch
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step(x)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    val = B * args.steps / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind,
                             "sample": f"{B} images/step x {args.steps} steps (the whole per-GPU batch of the workload), {what}, "
                                       f"torch {torch.__version__} CPU fp32, {cores} of {os.cpu_count()} host threads "
                                       f"(fastest of a small sweep)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------ our arm
def _pipeline_timer(dist, distributed, dev):
    """timed(stream, x, steps) -> ms for `steps` batches through a BatchStream (device events; max over ranks).  With a
    dict `last`, the results of the last batch are copied into it (as host tensors) after the timed region."""
    import torch

    def timed(stream, x, steps, last=None):
        stream.drain()
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream.compute)                       # everything idle here, so this is the start of the first batch
        for _ in range(steps):
            if stream._inflight == stream.depth:
                stream.collect()
            stream.submit(x)
        e1.record(stream.copy_out)                      # last stage of the last batch (stages of one slot run in order)
        while stream._inflight:                         # drain: the final collect() returns the last batch
            res = stream.collect()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if last is not None:
            gathered = res.pop("gathered", {})
            last.update({k: gathered.get(k, v).cpu() for k, v in res.items()})
        if distributed:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t.item())
        return ms
    return timed


def run_ours(args):
    import torch
    import torch.distributed as dist

    from dad_3dheads_b200 import _lib
    from dad_3dheads_b200.encoder_weights import synthetic_state_dict
    from dad_3dheads_b200.flame import load_flame_static
    from dad_3dheads_b200.predictor import DEFAULT_CONFIG, FaceMeshPredictor

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    distributed = world > 1
    if distributed:
        dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD if distributed else None

    # ---- constants: rank 0 owns them, everyone else receives them over NCCL (north_star: "NCCL broadcast of the bases")
    sd = synthetic_state_dict(0)
    static = load_flame_static()
    if distributed:
        from dad_3dheads_b200.distributed import broadcast_flame_static, broadcast_state_dict
        sd = broadcast_state_dict(sd, dev)
        static = broadcast_flame_static(static, dev)
    pred = FaceMeshPredictor(dict(DEFAULT_CONFIG), cuda_id=local_rank, state_dict=sd, precision=args.precision)
    if distributed:
        pred.head_mesh = type(pred.head_mesh)(pred.flame_constants, cuda_id=local_rank, static=static)

    B = args.batch
    subset = "445"
    g = torch.Generator().manual_seed(1234 + rank)
    # raw RGB frames as the reference's FaceMeshPredictor.__call__ takes them (uint8 HxWx3); the device-resident arm gets the
    # same batch already letter-boxed + normalised on the GPU (bit-identical to the reference's albumentations pipeline)
    x_host = torch.randint(0, 256, (B, 256, 256, 3), generator=g, dtype=torch.uint8).pin_memory()
    x_dev = pred.preprocess_batch(x_host)
    keys = ("3dmm_params", "points", "3d_vertices", "landmarks_445")
    timed = _pipeline_timer(dist, distributed, dev)

    def step_eager():
        return pred.predict_batch(x_dev, landmark_subset=subset)

    dev_stream = pred.open_stream(x_dev.shape, x_dev.dtype, landmark_subset=subset, keys=keys, host_results=False, group=group)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()                                 # sampled under load: warm-up + timed regions (same kernels)
    n_warm = max(args.warmup, 3)
    timed(dev_stream, x_dev, n_warm)
    launches0 = _lib.launch_count()
    step_eager()
    torch.cuda.synchronize()
    launches_per_step = _lib.launch_count() - launches0      # a graph replay launches the same kernels (counted at capture)
    last = {} if args.dump_outputs and rank == 0 else None
    ms_total = timed(dev_stream, x_dev, args.steps, last)    # EXACTLY K steps -> `value`
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    # a region of >= 1.5 s of the same steps: settled clocks, enough nvidia-smi samples; reported beside the K-step number
    per_step = ms_total / args.steps
    n_long = max(args.steps, int(1500.0 / max(per_step, 1e-3)) + 1) if not args.quick else args.steps
    n_long_t = torch.tensor([n_long], device=dev)
    if distributed:
        dist.broadcast(n_long_t, 0)
    n_long = int(n_long_t.item())
    ms_long = timed(dev_stream, x_dev, n_long)

    # N>1: the gathered buffers hold every rank's shard -- verify a checksum of each rank's slice against that rank's own
    gather_check = None
    if distributed:
        dev_stream.submit(x_dev)
        res = dev_stream.collect()
        torch.cuda.synchronize()
        mine = torch.stack([res[k].double().sum() for k in dev_stream.gather_keys])             # [3]
        allsums = torch.empty(world, mine.numel(), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(allsums, mine)
        ok = True
        for j, k in enumerate(dev_stream.gather_keys):
            gk = res["gathered"][k]
            for r in range(world):
                sl = gk[r * B:(r + 1) * B].double().sum()
                ok = ok and bool(sl == allsums[r, j])
            ok = ok and bool(torch.equal(gk[rank * B:(rank + 1) * B], res[k]))
        okt = torch.tensor([1 if ok else 0], device=dev)
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
        gather_check = bool(okt.item())

    # per-kernel timing for the roofline: the same step, launched eagerly with CUDA events around every tile-engine launch
    torch.cuda.synchronize()
    pred.model.set_profile(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_prof = min(args.steps, 10)
    e0.record()
    for _ in range(n_prof):
        step_eager()
    e1.record()
    torch.cuda.synchronize()
    ms_eager = e0.elapsed_time(e1)
    lay = pred.model.profile_layers()
    algo_bytes_per_launch = sum(l["bytes"] for l in lay) / max(len(lay), 1)
    prof = pred.model.profile_read()
    pred.model.set_profile(False)

    # end to end through the public pipelined API: pinned host frames in, pinned host results out, copies inside the region
    e2e_stream = pred.open_stream(x_host.shape, x_host.dtype, landmark_subset=subset, keys=keys, host_results=True, group=group)
    timed(e2e_stream, x_host, 3)
    ms_e2e = timed(e2e_stream, x_host, args.steps)
    ms_e2e_long = timed(e2e_stream, x_host, n_long)
    clocks = sampler.stop() if sampler else None
    # the un-pipelined latency of one step (H2D -> graph -> [all-gather] -> D2H -> sync), for reference
    e2e_stream.submit(x_host); e2e_stream.collect()
    t0 = time.perf_counter()
    for _ in range(5):
        e2e_stream.submit(x_host)
        e2e_stream.collect()
    serial_ms = (time.perf_counter() - t0) / 5 * 1e3
    host_out = e2e_stream.slots[0]["host"]

    if rank == 0:
        peaks = _peaks()
        heads = B * world * args.steps
        value = heads / (ms_total * 1e-3)
        e2e_value = heads / (ms_e2e * 1e-3)
        gemm_ms, gemm_launches, useful_flops = prof
        products = PRODUCTS[args.precision]
        achieved = useful_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
        peak = peaks["bf16_tflops_sustained"]
        traffic, traffic_src = _traffic_from_profile()
        h2d = x_host.numel() * x_host.element_size()
        d2h = sum(v.numel() * v.element_size() for v in host_out.values())
        cfg = workload_config(args, world)
        cfg.update({"decode": "flame_decode_kernel (the batched API's default): one fp16 product per MAC, template exact in two K "
                              "columns, fp32 accumulate -- vertices relL2 3.5e-5 vs the reference (contract 1e-4, see parity) + LBS + "
                              "projection + 445-landmark gather; the strict run (strict_fp32_operands) uses the same decode",
                    "parallelism": (f"dp{world} (batch sharded, NCCL bcast constants at start-up, per-step all-gather of params/"
                                    f"vertices/landmarks on a side stream overlapping the next step)") if distributed
                    else "single GPU",
                    "l2": "no explicit flush: per-step working set (50 MB input + >1 GB activations) exceeds the 126 MB L2"})
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": DTYPE[args.precision],
            "data": "synthetic",
            "config": cfg,
            "sustained": {"value": B * world * n_long / (ms_long * 1e-3), "unit": UNIT, "steps": n_long,
                          "seconds": ms_long * 1e-3, "e2e_value": B * world * n_long / (ms_e2e_long * 1e-3),
                          "note": "the same step over a >= 1.5 s timed region (value above is EXACTLY --steps steps)"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps, "serial_latency_ms": serial_ms,
                    "api": "FaceMeshPredictor.open_stream(...).submit(uint8 [B,256,256,3] pinned host frames) / .collect() -> "
                           "pinned host params/points/vertices/landmarks; letter-box + normalise on the GPU; two slots: H2D of "
                           "batch i+1 and D2H of batch i-1 run on copy streams beside the graph replay of batch i"},
            "gpu_launches": int(launches_per_step * args.steps),
            "launch_mode": "CUDA graph replay of FaceMeshPredictor.predict_batch (one graph launch per step; gpu_launches = "
                           "kernels inside the graph x steps)",
            "clocks": clocks,
            "roofline": {"kernel": "tile_gemm_kernel<EpiConv> (all conv/linear layers, tcgen05)", "bound": "tensor",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                         "traffic": traffic if B == 64 and args.precision == "fp16x2" else None,
                         "traffic_unit": "DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, averaged "
                                         "over the tile-engine launches of one step)", "traffic_source": traffic_src,
                         "algorithmic_bytes_per_launch": algo_bytes_per_launch,
                         "peak_source": peaks["source"] + " bf16 dense, sustained",
                         "products_per_mac": products, "executed_tflops": achieved * products,
                         "frac_executed": achieved * products / peak if peak else None,
                         "kernel_ms_per_step": gemm_ms / n_prof, "launches_per_step": gemm_launches / n_prof,
                         "share_of_step": gemm_ms / ms_eager if ms_eager else None,
                         "measured_in": "an EAGER pass of the same step after the timed region (CUDA events around every "
                                        "tile-engine launch, so each launch's latency is inside its interval; slightly longer "
                                        f"than the graph-replayed step: {ms_eager / n_prof:.3f} ms/step eager)",
                         "algorithmic_gflop_per_head": useful_flops / (B * n_prof) / 1e9},
        }
        if gather_check is not None:
            line["gather_verified"] = gather_check
        print_later = line
    del dev_stream, e2e_stream

    # ---- sub-objects (bounded; none of them inside the headline's timed regions)
    extras = {}
    if world == 1 and args.precision != "fp32" and not args.no_strict:
        # the same step with strict 24-bit operands (bf16x3, 6 products), device-resident, for comparison
        strict = FaceMeshPredictor(dict(DEFAULT_CONFIG), cuda_id=local_rank, state_dict=sd, precision="fp32")
        st = strict.open_stream(x_dev.shape, x_dev.dtype, landmark_subset=subset, keys=keys, host_results=False)
        timed(st, x_dev, 3)
        n_s = max(3, args.steps // 2)
        ms_s = timed(st, x_dev, n_s)
        extras["strict_fp32_operands"] = {"value": B * n_s / (ms_s * 1e-3), "unit": UNIT, "ms_per_step": ms_s / n_s,
                                          "steps": n_s, "mode": DTYPE["fp32"]}
        del strict, st
    if not args.no_extras and args.config == 2:
        if world == 1:
            extras["decode_microbench"] = decode_microbench(pred.head_mesh, dev, steps=2, warmup=1, n_total=1 << 20)
            torch.cuda.empty_cache()
            extras["config3"] = sub_pipeline(FaceMeshPredictor, DEFAULT_CONFIG, sd, None, local_rank, 512, "bf16", timed,
                                             None, 1, "configs[2]: batch 512, bf16 encoder / fp32-class FLAME decode + "
                                             "445-landmark projection, 1 GPU")
        else:
            del pred
            torch.cuda.empty_cache()
            extras["config4"] = sub_pipeline(FaceMeshPredictor, DEFAULT_CONFIG, sd, static, local_rank, 512, args.precision,
                                             timed, group, world, f"configs[3]: batch {512 * world} = {world} x 512 sharded, "
                                             "NCCL all-gather of params/vertices/landmarks overlapped with the next step")
    if rank == 0:
        line = print_later
        line.update(extras)
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_baseline(sd, parity_with=pred)
            line["parity"] = cb.pop("parity", None)
            line["cpu_baseline"] = cb
        print(json.dumps(line), flush=True)
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def sub_pipeline(FaceMeshPredictor, DEFAULT_CONFIG, sd, static, local_rank, B, precision, timed, group, world, what):
    """A short device-resident + end-to-end measurement of another BASELINE config with the same machinery."""
    import torch
    pred = FaceMeshPredictor(dict(DEFAULT_CONFIG), cuda_id=local_rank, state_dict=sd, precision=precision)
    if static is not None:
        pred.head_mesh = type(pred.head_mesh)(pred.flame_constants, cuda_id=local_rank, static=static)
    g = torch.Generator().manual_seed(99 + int(os.environ.get("RANK", "0")))
    x_host = torch.randint(0, 256, (B, 256, 256, 3), generator=g, dtype=torch.uint8).pin_memory()
    x_dev = pred.preprocess_batch(x_host)
    keys = ("3dmm_params", "points", "3d_vertices", "landmarks_445")
    st = pred.open_stream(x_dev.shape, x_dev.dtype, landmark_subset="445", keys=keys, host_results=False, group=group)
    timed(st, x_dev, 3)
    n = 8
    ms = timed(st, x_dev, n)
    del st
    st = pred.open_stream(x_host.shape, x_host.dtype, landmark_subset="445", keys=keys, host_results=True, group=group)
    timed(st, x_host, 2)
    ms_e = timed(st, x_host, n)
    out = {"workload": what, "per_gpu_batch": B, "global_batch": B * world, "encoder_precision": precision, "steps": n,
           "value": B * world * n / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / n,
           "e2e_value": B * world * n / (ms_e * 1e-3), "e2e_ms_per_step": ms_e / n}
    del st, pred
    torch.cuda.empty_cache()
    return out


def decode_microbench(head_mesh, dev, steps, warmup, n_total=1 << 20, fast=True, cluster=False, last=None):
    """BASELINE.json configs[4]: FLAME-decode-only, `n_total` param vectors -> 5023-vertex meshes per step, streamed through a
    fixed output ring; reports the blend-shape tensor-core roofline and the HBM-write roofline side by side.  With a dict
    `last`, the vertices of the last pass of the last step are copied into it after the timed region."""
    import torch
    from dad_3dheads_b200 import _lib
    from oracle.flame_oracle import sample_params                   # input generation only (outside the timed region)
    dec = head_mesh.flame.decoder(dev)
    chunk = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * 4
    base = sample_params(8192, seed=0).to(dev)
    params = base.repeat(n_total // 8192, 1)                        # n_total x 413 (1.7 GB at 1M), seeded
    passes = [(i, min(i + chunk, n_total)) for i in range(0, n_total, chunk)]

    def step():
        for lo, hi in passes:
            v3, _ = dec.decode(params[lo:hi], want_vertices=True, want_projected=False, fast=fast, cluster=cluster)
        return v3

    for _ in range(max(warmup, 1)):
        step()
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps - 1):
        step()
    v3 = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if last is not None:
        last["3d_vertices"] = v3
    del v3
    value = n_total * steps / (ms * 1e-3)
    peaks = _peaks()
    products = 1 if fast else 3
    achieved = value * FLOPS_PER_HEAD_BLEND / 1e12
    peak = peaks["bf16_tflops_sustained"]
    del params
    return {"metric": "heads/sec FLAME decode only (413 params -> 5023x3 vertices)", "value": value, "unit": UNIT,
            "steps": steps, "heads_per_step": n_total, "heads_per_pass": chunk, "ms_per_step": ms / steps,
            "dtype": "fp16 operands (1 product), template exact in two K columns, fp32 accumulate" if fast else
                     "fp16 hi/lo split operands (3 products), fp32 accumulate",
            "gpu_launches": int(_lib.launch_count() - l0),
            "roofline": {"kernel": "flame decode (blend shapes + skinning + rotation, fused)", "bound": "tensor",
                         "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "peak_source": peaks["source"] + " 16-bit dense, sustained", "products_per_mac": products,
                         "executed_tflops": achieved * products, "frac_executed": achieved * products / peak,
                         "hbm_gbs_algorithmic": value * BYTES_PER_HEAD_DECODE / 1e9,
                         "hbm_frac": value * BYTES_PER_HEAD_DECODE / 1e9 / peaks["hbm_gbs"]}}


def run_decode_microbench(args):
    """`--config 5` as its own bench line."""
    import torch
    from dad_3dheads_b200 import HeadMesh
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    hm = HeadMesh(cuda_id=0)
    sampler = ClockSampler(0)
    sampler.start()
    fast = args.precision in ("fp16", "bf16")
    last = {} if args.dump_outputs else None
    d = decode_microbench(hm, dev, args.steps, max(args.warmup, 3), n_total=args.batch, fast=fast, cluster=args.decode_cluster,
                          last=last)
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    clocks = sampler.stop()
    line = {"metric": d.pop("metric"), "value": d["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": d["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": d["dtype"], "data": "synthetic",
            "config": {"workload": f"{CONFIGS[5]['base']} -- {args.batch} heads per step", "heads_per_step": args.batch,
                       "heads_per_pass": d["heads_per_pass"], "output": "vertices [pass,5023,3] fp32 ring buffer "
                       "(overwritten every pass)", "l2": "outputs (910 MB per pass) exceed L2"},
            "gpu_launches": d["gpu_launches"], "clocks": clocks, "roofline": d["roofline"]}
    print(json.dumps(line), flush=True)


def cpu_baseline(sd, parity_with=None):
    """The reference's CPU path (kind "reference": the unmodified reference code through oracle/ref_harness.py; "port": the
    oracle restatement when oracle/_ref is absent) timed on this box's host cores on a bounded sample; with parity_with = a
    FaceMeshPredictor it also checks that predictor's outputs on the sample against it."""
    import torch
    step, what, kind = _reference_runner(sd)
    sample = 16
    x = torch.randn(sample, 3, 256, 256, generator=torch.Generator().manual_seed(0))
    cores = _best_threads_fn(step, x[:4])
    step(x)
    reps = 0
    t0 = time.perf_counter()
    while reps < 3 or (time.perf_counter() - t0 < 12.0 and reps < 40):
        step(x)
        reps += 1
    dt = time.perf_counter() - t0
    out = {"value": sample * reps / dt, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"{reps} passes of {sample} images (encoder + FLAME decode x2 + projection + 445 take), {what}, torch "
                     f"{torch.__version__} CPU fp32, {cores} of {os.cpu_count()} host threads (fastest of a small sweep)"}
    if parity_with is not None:
        ref = step(x)
        got = parity_with.predict_batch(x, landmark_subset="445")

        def rel(k):
            a, b = got[k].double().cpu(), ref[k].double().cpu()
            return float((a - b).norm() / b.norm())
        v_l2 = float((got["3d_vertices"].double().cpu() - ref["3d_vertices"].double()).norm(dim=-1).max())
        out["parity"] = {"params_rel_l2": rel("3dmm_params"), "vertices_rel_l2": rel("3d_vertices"),
                         "landmarks_445_rel_l2": rel("landmarks_445"), "vertex_l2_max_m": v_l2, "tolerance": 1e-4,
                         "against": f"{what}, fp32 on the CPU, same {sample} images"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5],
                    help="BASELINE.json config, 1-based as in SURVEY §8(d): 2 = configs[1] (headline, default), 3 = batch 512 "
                         "bf16 encoder, 4 = 512 per GPU across N GPUs, 5 = decode-only microbench")
    ap.add_argument("--batch", type=int, default=None, help="images per GPU per step (default: the config's)")
    ap.add_argument("--precision", default=None, choices=["fp32", "bf16x3", "fp16x2", "bf16x2", "fp16", "bf16"])
    ap.add_argument("--decode-cluster", action="store_true", help="decode microbench: 2x2 multicast clusters (A/B only)")
    ap.add_argument("--no-strict", action="store_true", help="skip the strict-operand comparison run")
    ap.add_argument("--no-extras", action="store_true", help="skip the decode_microbench / config3 / config4 sub-objects")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="profiling aid (ncu launch lists): no >= 1.5 s region, no sub-objects, "
                    "no strict-mode run, no CPU baseline -- only warm-up + the K timed steps of both arms")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (at most 64 MB; a seeded row sample "
                         "of larger outputs)")
    ap.add_argument("--workload", default=None, choices=["pipeline", "decode"], help="legacy alias: decode = --config 5")
    args = ap.parse_args()
    if args.workload == "decode":
        args.config = 5
    args = resolve(args)
    if args.quick:
        args.no_extras = args.no_strict = args.no_cpu_baseline = True
    if args.impl == "reference":
        run_reference(args)
    elif args.config == 5:
        run_decode_microbench(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
