#!/usr/bin/env python
"""bench.py -- pose hypotheses / second through render + coarse + 5x refine (BASELINE.json metric).

    python bench.py --gpus 1 --steps 5 --warmup 3            # this framework (libmpx.so, sm_100a)
    python bench.py --impl reference --steps 2 --warmup 1    # the reference path on the host cores (CPU oracle port)
    python bench.py --impl torch-gpu                         # the same networks through stock torch / cuDNN on this GPU
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ... [--scaling strong]

Workload (config.workload): BASELINE.json configs[1] "megapose-1.0-RGB: 1 object x 576 coarse hypotheses + 5
refiner iters" at the reference's 240x320 render size (--render-size 224x224 for the size the metric's text names),
synthetic 480x640 frame, procedural 10k-triangle mesh, seeded random vanilla_resnet34 weights in the model-zoo
checkpoint format (workloads/scenes.py: bench_scene).  One step = one frame through PoseEstimator's inference pipeline.
Frames are fed the way a stream of frames is served (--frames-in-flight 2, megapose6d_b200/frame_pipeline.py): two
estimators on two CUDA streams, the latency-bound refiner iterations of frame i beside the coarse stage of frame i+1;
every frame's result is produced and read exactly as by run_inference_pipeline (bit-identical, tested).  The line also
carries `single_frame`: the same K steps with one blocking run_inference_pipeline call after the other.
Weak scaling (default): a frame with one detection per rank, rows sharded by detection, one all-gather per stage.
Strong scaling (--scaling strong): ONE frame (1 x 576, or --workload ycbv21: 21 x 576 = BASELINE configs[3]) whose
rows are split over the N ranks.  The detection boxes change from step to step (a pool of jittered boxes), so a timed
step is never a replay of identical inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

M_GRID = 576
N_REFINER_ITERS = 5
# SURVEY.md 8(d), FLOP = 2*MAC, conv + linear: {render size: (coarse/scoring forward, RGB refiner forward)} GFLOP per sample
GFLOP = {(240, 320): (12.068, 14.236), (224, 224): (7.799, 9.215)}
# 16-bit bytes the 36 convolutions of one coarse forward move at least once per hypothesis at 240x320 (each conv: input
# read + output write + residual read; weights excluded): stem 2.46 MB in + 0.61 MB pooled out (the max-pool runs in its
# epilogue; 2 x 2.46 MB before), layer1 6 convs of 60x80x64, ... = 26.42 MB
ALGO_CONV_BYTES_PER_HYP = 26.42e6


def gflop_per_hyp(render_size, n_det=1):
    c, r = GFLOP[tuple(render_size)]
    return c + (N_REFINER_ITERS * r + c) / M_GRID  # config-2 unit: coarse + (5 refiner + 1 scoring forward) / 576


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="mpx", choices=["mpx", "reference", "torch-gpu"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--workload", default="rgb576", choices=["rgb576", "ycbv21"])
    ap.add_argument("--render-size", default="240x320")
    ap.add_argument("--frames-in-flight", type=int, default=2, help="1: one blocking run_inference_pipeline call per step")
    ap.add_argument("--overlap-heads", action="store_true", help="A/B: do not gate a frame's coarse stage on its predecessor's")
    ap.add_argument("--reserve-sms", type=int, default=-1, help="size the persistent grids for (SMs - N): SMs left to the "
                                                                "latency-bound tail of the other frame in flight (-1: default)")
    ap.add_argument("--cpu-sample", type=int, default=32, help="coarse hypotheses in one bounded CPU step")
    ap.add_argument("--no-full-unit", action="store_true", help="CPU arm: skip the one complete 576-hypothesis unit")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (final poses and per-detection scores) as DIR/<name>.npy")
    a = ap.parse_args()
    a.render_size = tuple(int(v) for v in a.render_size.lower().split("x"))
    assert a.render_size in GFLOP, f"--render-size must be one of {sorted(GFLOP)}"
    return a


def build_scene(args, n_ranks: int):
    from workloads import scenes

    if args.workload == "ycbv21":
        assert args.scaling == "strong" or n_ranks == 1, "ycbv21 is a single-frame (strong-scaling) workload"
        return scenes.ycbv_scene(21)
    return scenes.bench_scene(1 if args.scaling == "strong" else n_ranks, render_size=args.render_size)


def workload_config(args, sc, n_gpus: int):
    h, w = sc["render_size"]
    B = len(sc["labels"])
    return {"workload": f"{sc['model']}: {B} object(s) x {M_GRID} coarse hypotheses + {N_REFINER_ITERS} refiner iters + "
                        f"scoring per frame (BASELINE configs[{3 if args.workload == 'ycbv21' else 1}]); 480x640 frame, "
                        f"{h}x{w} crops/renders, 10k-triangle procedural meshes, vanilla_resnet34 random weights",
            "hypotheses_per_step": M_GRID * B, "scaling": args.scaling,
            "parallelism": f"hypothesis rows sharded x{n_gpus}" + (" (one detection per rank)" if args.scaling == "weak" else
                                                                  " (one frame over all ranks)"),
            "inputs": "detection boxes jittered per step (pool of 4)",
            "frames_in_flight": f"{max(1, args.frames_in_flight)} (megapose6d_b200/frame_pipeline.py: the refiner iterations of "
                                "frame i overlap the coarse stage of frame i+1 on a second stream; every frame's result is "
                                "produced and read; `single_frame` has the one-blocking-call-per-step numbers)",
            "l2": f"network input tensor ({2 * 64 * (h // 2) * (w // 2) * M_GRID * B / n_gpus / 1e9:.2f} GB per rank and "
                  "step) >> 126 MB L2, no explicit flush"}


def bbox_pool(bboxes, n=4):
    """Jittered copies of the detection boxes (+-2 px, seeded): same hypothesis count, different numbers every step."""
    import torch

    g = torch.Generator().manual_seed(7)
    return [bboxes + (0.0 if i == 0 else 1.0) * (4.0 * torch.rand(bboxes.shape, generator=g) - 2.0) for i in range(n)]


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path on the host cores (kind "port": the Python reference cannot be
# compiled into oracle/_ref, and Panda3D is absent, so torch fp32 + the C rasteriser of oracle/raster_ref.c stand in)
# ---------------------------------------------------------------------------------------------
def cpu_estimator(sc, cores):
    import torch

    from oracle import pipeline_ref
    from tests import helpers
    from workloads import weights

    torch.set_num_threads(cores)
    meshes = helpers.ref_meshes_from_dataset(sc["ds"])
    rr = pipeline_ref.RefRenderer(meshes, n_threads=cores)
    oc = pipeline_ref.RefPosePredictor(sc["sd_coarse"], weights.COARSE_CFG, meshes, rr, render_size=sc["render_size"])
    orf = pipeline_ref.RefPosePredictor(sc["sd_refiner"], sc["cfg_refiner"], meshes, rr, render_size=sc["render_size"])
    return pipeline_ref.RefPoseEstimator(oc, orf, bsz_images=128, bsz_objects=8, SO3_grid_size=M_GRID)


def cpu_unit(est, sc, n_coarse: int):
    """One pass of the path on the host for one detection: n_coarse coarse hypotheses (576 = the complete unit), then 5
    refiner iterations and the scoring pass on the best one.  Returns (seconds of the coarse part, seconds of the rest)."""
    import torch

    df1 = sc["det_df"].iloc[:1].copy()
    images, K, bboxes = sc["images"], sc["K"], sc["bboxes"]
    with torch.no_grad():
        t0 = time.time()
        df_c, TCO_c = est.forward_coarse_model(images, K, df1, bboxes[:1], max_hypotheses=n_coarse)
        t_coarse = time.time() - t0
        keep = est.filter_pose_estimates(df_c, 1, "coarse_logit")
        t0 = time.time()
        ref = est.forward_refiner(images, K, df_c.iloc[keep].reset_index(drop=True), TCO_c[keep], N_REFINER_ITERS)
        est.forward_scoring_model(images, K, df_c.iloc[keep].reset_index(drop=True), ref[f"iteration={N_REFINER_ITERS}"]["TCO_output"])
        t_refine = time.time() - t0
    return t_coarse, t_refine


def run_reference_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch

    sc = build_scene(args, 1)
    # torch's CPU convolutions stop scaling (and regress) past a few dozen threads at these batch sizes
    cores = min(os.cpu_count() or 1, 32)
    est = cpu_estimator(sc, cores)
    with torch.no_grad():
        est.forward_coarse_model(sc["images"], sc["K"], sc["det_df"].iloc[:1].copy(), sc["bboxes"][:1], max_hypotheses=2)  # op loading
    for _ in range(max(0, args.warmup)):
        cpu_unit(est, sc, max(4, args.cpu_sample // 4))
    vals, secs = [], []
    for _ in range(max(1, args.steps)):
        tc, tr = cpu_unit(est, sc, args.cpu_sample)
        vals.append(M_GRID / (M_GRID * tc / args.cpu_sample + tr))
        secs.append(tc + tr)
    sampled = float(np.mean(vals))
    sample = (f"{args.steps} steps of {args.cpu_sample} of 576 coarse hypotheses + 5 refiner iterations and scoring of the best "
              f"one, extrapolated to the 576-hypothesis unit: {sampled:.2f} hyp/s")
    value = sampled
    if not args.no_full_unit:
        tc, tr = cpu_unit(est, sc, M_GRID)
        value = M_GRID / (tc + tr)
        sample = (f"one COMPLETE unit, not extrapolated: 576 coarse hypotheses ({tc:.1f} s) + 5 refiner iterations and scoring "
                  f"({tr:.2f} s); " + sample)
    sample += f"; torch fp32 + C rasteriser on {cores} threads"
    line = {
        "metric": "pose hypotheses/sec through render+coarse+5x refine", "value": value, "unit": "hypotheses/s",
        "impl": "reference", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 * float(np.mean(secs)), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, sc, 1),
        "cpu_baseline": {"value": value, "unit": "hypotheses/s", "cores": cores, "kind": "port", "sample": sample,
                         "sampled_value": sampled},
        "e2e": {"value": value, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def cpu_baseline_subprocess(args):
    """The CPU leg of the mpx arm runs in its own process: nothing of oracle/ is loaded into the measured process."""
    cmd = [sys.executable, str(Path(__file__).resolve()), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--cpu-sample", str(args.cpu_sample), "--render-size", "x".join(map(str, args.render_size))]
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env)
        line = next(l for l in reversed(res.stdout.splitlines()) if l.startswith("{"))
        return json.loads(line)["cpu_baseline"]
    except Exception as exc:  # noqa: BLE001 -- the baseline is a report, never a reason to lose the bench line
        return {"value": None, "unit": "hypotheses/s", "cores": 0, "kind": "port", "sample": f"failed: {exc!r}"[:300]}


# ---------------------------------------------------------------------------------------------
# torch / cuDNN arm: the same two networks through stock PyTorch on this GPU (the "existing Blackwell kernel" bar)
# ---------------------------------------------------------------------------------------------
def torch_gpu_baseline(sc, quick: bool = False):
    """Network-only time of one config-2 unit through torch / cuDNN: coarse forward over 576 hypotheses (one batch, and in
    the reference's chunks of bsz_images = 128), 5 refiner forwards and one scoring forward at batch 1 (eager and as CUDA
    graphs).  No rendering, crops or host bookkeeping: an UPPER bound on what a torch-on-GPU pipeline could reach."""
    import torch

    from workloads import torch_resnet as T

    h, w = sc["render_size"]
    out = {"unit": "ms", "what": "coarse forward x576 | refiner forward x1 | unit = coarse576 + 5 refiner + 1 scoring forward"}
    for prec in T.PRECISIONS:
        if quick and prec not in ("fp32_strict", "fp16_channels_last"):
            continue
        c576 = min(T.time_forward(sc["sd_coarse"], M_GRID, h, w, prec), T.time_forward(sc["sd_coarse"], M_GRID, h, w, prec, chunk=128))
        r1 = T.time_forward(sc["sd_refiner"], 1, h, w, prec, iters=10, graph=True)
        s1 = T.time_forward(sc["sd_coarse"], 1, h, w, prec, iters=10, graph=True)
        unit_ms = c576 + N_REFINER_ITERS * r1 + s1
        out[prec] = {"coarse576_ms": c576, "refiner1_ms": r1, "scoring1_ms": s1, "unit_ms": unit_ms,
                     "hyp_per_s_network_only": M_GRID / unit_ms * 1e3,
                     "coarse_tflops": GFLOP[(h, w)][0] * M_GRID / c576}
        torch.cuda.empty_cache()
    return out


def run_torch_gpu_arm(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch

    assert torch.cuda.is_available()
    sc = build_scene(args, 1)
    base = torch_gpu_baseline(sc)
    best = min((k for k in base if isinstance(base[k], dict)), key=lambda k: base[k]["unit_ms"])
    line = {"metric": "pose hypotheses/sec through render+coarse+5x refine", "impl": "torch-gpu",
            "value": base[best]["hyp_per_s_network_only"], "unit": "hypotheses/s", "n_gpus": 1, "steps": 5, "warmup": 3,
            "ms_per_step": base[best]["unit_ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": best, "data": "synthetic", "config": workload_config(args, sc, 1),
            "note": "network forwards only (no rendering / crops / bookkeeping): an upper bound for a torch-on-GPU pipeline",
            "gpu_torch_baseline": base}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def host_outputs(final):
    """What run_inference_pipeline hands its caller for one frame, as host arrays: every tensor of the final collection
    and every numeric column of its infos (one row per detection), in float32 or float64."""
    out = {}
    for name, t in final.tensors.items():
        a = t.detach().cpu().numpy()
        out[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    for col in final.infos.columns:
        v = final.infos[col].to_numpy()
        if np.issubdtype(v.dtype, np.number) or v.dtype == np.bool_:
            out[f"infos_{col}"] = v if v.dtype in (np.float32, np.float64) else v.astype(np.float64)
    return out


def write_outputs(outputs, out_dir: Path):
    total = sum(a.nbytes for a in outputs.values())
    assert total <= 64 << 20, f"{total} bytes of outputs exceed the 64 MB dump limit"
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in outputs.items():
        np.save(out_dir / f"{name}.npy", a)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_mpx_arm(args):
    import ctypes

    import torch
    import torch.distributed as dist

    from megapose6d_b200 import _abi
    from megapose6d_b200.parallel import HypothesisSharder
    from megapose6d_b200.tensor_collection import PandasTensorCollection
    from megapose6d_b200.types import ObservationTensor
    from workloads import scenes

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py --impl mpx needs a CUDA device (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n_gpus = world
    sc = build_scene(args, n_gpus)
    images, K, det_df = sc["images"], sc["K"], sc["det_df"]
    from megapose6d_b200.frame_pipeline import FramePipeline

    n_fif = max(1, args.frames_in_flight)
    if args.reserve_sms >= 0:
        from megapose6d_b200 import frame_pipeline as _fp

        _fp.set_reserved_sms(args.reserve_sms)
    ests = [scenes.build_estimator(sc, sharder=HypothesisSharder(enabled=world > 1)) for _ in range(n_fif)]
    est = ests[0]
    pipe = FramePipeline(None, estimators=ests, serialize_heads=not args.overlap_heads) if n_fif > 1 else None
    lib = _abi.lib()
    n_det = len(sc["labels"])
    h, w = sc["render_size"]

    pool = bbox_pool(sc["bboxes"])
    images_dev, K_dev, pool_dev = images.cuda(), K.cuda(), [b.cuda() for b in pool]
    images_pin, K_pin, pool_pin = images.pin_memory(), K.pin_memory(), [b.pin_memory() for b in pool]
    counter = [0]

    kw = dict(n_refiner_iterations=N_REFINER_ITERS, n_pose_hypotheses=1)

    def frame_device():
        counter[0] += 1
        return ObservationTensor(images_dev, K_dev), PandasTensorCollection(det_df.copy(), bboxes=pool_dev[counter[0] % len(pool_dev)])

    def frame_host():  # this step's inputs from pinned host memory
        counter[0] += 1
        obs = ObservationTensor(images_pin.cuda(non_blocking=True), K_pin.cuda(non_blocking=True))
        return obs, PandasTensorCollection(det_df.copy(), bboxes=pool_pin[counter[0] % len(pool_pin)].cuda(non_blocking=True))

    def read_back(final):  # the step's result on the host
        return final.poses.cpu(), final.infos["pose_score"].values

    last = [None]  # the final collection of the most recent step (for --dump-outputs)

    def step_device(e=None):
        obs, det = frame_device()
        last[0] = (e or est).run_inference_pipeline(obs, detections=det, **kw)[0]
        return last[0]

    def run_single(steps, host: bool):  # one blocking call per step
        for _ in range(steps):
            if host:
                obs, det = frame_host()
                read_back(est.run_inference_pipeline(obs, detections=det, **kw)[0])
            else:
                step_device()

    def run_in_flight(steps, host: bool):  # the same steps through the frame pipeline; every result is collected
        n_done = 0
        for _ in range(steps):
            done = pipe.submit(*(frame_host() if host else frame_device()), **kw)
            if done is not None:
                n_done += 1
                last[0] = done[0]
                if host:
                    read_back(done[0])
        for done in pipe.drain():
            n_done += 1
            last[0] = done[0]
            if host:
                read_back(done[0])
        pipe.join()
        assert n_done == steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, host):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(steps, host)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    warmup = max(3, args.warmup)
    for e in ests:
        for _ in range(warmup + 2):  # first sight runs eagerly, the second captures the graphs, later ones replay
            step_device(e)
    run = run_in_flight if pipe is not None else run_single
    run(2 * n_fif, False)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms = timed(run, args.steps, False)
    # copied out before later steps reuse the estimators' static buffers
    outputs = host_outputs(last[0]) if args.dump_outputs else None
    run(2 * n_fif, True)
    e2e_ms = timed(run, args.steps, True)
    single = None
    if pipe is not None:  # the same steps, one blocking run_inference_pipeline call after the other
        run_single(2, False)
        s_ms = timed(run_single, args.steps, False)
        run_single(2, True)
        s_e2e_ms = timed(run_single, args.steps, True)
        single = (s_ms, s_e2e_ms)
    clocks = sampler.stop() if rank == 0 else None  # sampled over all timed regions (device-resident and end-to-end)

    # roofline of the dominant kernels (the convolutions of the coarse forward): CUDA events around every conv launch, same
    # workload.  The coarse forward normally replays a CUDA graph (its launches cannot be timed one by one), so for this
    # pass it is launched eagerly; the small-batch forwards (<= 64 rows) keep replaying graphs.
    saved_gmb = est.coarse_model.graph_max_batch
    est.coarse_model.graph_max_batch = 64
    lib.mpx_profile_enable(1)
    prof_steps = 2
    for _ in range(prof_steps):
        step_device()
    conv_ms, conv_fl, conv_n = ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    _abi.check(lib.mpx_profile_summary(ctypes.byref(conv_ms), ctypes.byref(conv_fl), ctypes.byref(conv_n)))
    lib.mpx_profile_enable(0)
    est.coarse_model.graph_max_batch = saved_gmb
    # kernels of libmpx.so per step: counted on one step launched eagerly (graph replays execute the same kernels but do
    # not pass through the library's launch counter)
    flags = (est.coarse_model.use_cuda_graphs, est.refiner_model.use_cuda_graphs)
    est.coarse_model.use_cuda_graphs = est.refiner_model.use_cuda_graphs = False
    lib.mpx_net_set_graphs(0)
    l0 = lib.mpx_launch_count()
    step_device()
    torch.cuda.synchronize()
    launches = torch.tensor([(lib.mpx_launch_count() - l0) * args.steps], device="cuda", dtype=torch.float64)
    lib.mpx_net_set_graphs(1)
    est.coarse_model.use_cuda_graphs, est.refiner_model.use_cuda_graphs = flags
    if world > 1:
        dist.all_reduce(launches)
    barrier()

    del pipe
    hyp_per_step = M_GRID * n_det
    ms_per_step = total_ms / args.steps
    value = hyp_per_step / (ms_per_step / 1000.0)
    e2e_value = hyp_per_step / (e2e_ms / args.steps / 1000.0)
    if rank == 0:
        peaks_path = ROOT / "MEASURED_PEAKS.json"
        if peaks_path.exists():
            peaks = json.loads(peaks_path.read_text())
            burst, sustained = float(peaks.get("bf16_tflops", 1700.0)), float(peaks.get("bf16_tflops_sustained", 1400.0))
            peak_src = "MEASURED_PEAKS.json bf16_tflops (burst: the timed region is a sub-second burst at full clocks)"
        else:
            burst, sustained = 1700.0, 1400.0
            peak_src = "fallback figures of B200_PROFILING.md (MEASURED_PEAKS.json absent)"
        conv_ms_per_step = conv_ms.value / prof_steps
        # The event-timed launches are the convolutions of this rank's coarse forward(s) (the refiner iterations and the
        # final scoring replay CUDA graphs, whose kernels are not individually timed): algorithmic work of exactly those
        # launches = rows x GFLOP of one coarse forward (SURVEY 8d, FLOP = 2*MAC)
        rows_rank = M_GRID * n_det / n_gpus
        algo_tflop_per_step = GFLOP[(h, w)][0] * rows_rank / 1000.0
        achieved = algo_tflop_per_step / (conv_ms_per_step / 1000.0)
        traffic = None
        tpath = ROOT / "profiles" / "conv_traffic.json"
        if tpath.exists() and (h, w) == (240, 320) and rows_rank == M_GRID:
            # dram__bytes_read.sum + dram__bytes_write.sum of the same 36 launches from one ncu pass of this workload (a
            # constant read from the file, not a measurement of this run)
            tj = json.loads(tpath.read_text())
            traffic = float(tj["dram_read_bytes"]) + float(tj["dram_write_bytes"])
        line = {
            "metric": "pose hypotheses/sec through render+coarse+5x refine", "value": value, "unit": "hypotheses/s",
            "impl": "mpx", "n_gpus": n_gpus, "steps": args.steps, "warmup": warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f16" if lib.mpx_act_dtype() == 0 else "bf16", "data": "synthetic",
            "config": workload_config(args, sc, n_gpus),
            "e2e": {"value": e2e_value, "unit": "hypotheses/s",
                    "h2d_bytes_per_step": int(images.numel() * 4 + K.numel() * 4 + sc["bboxes"].numel() * 4),
                    "d2h_bytes_per_step": int(n_det * 16 * 4 + n_det * 4 * 2 + M_GRID * n_det * 8 * 3)},
            "gpu_launches": int(launches.item()),
            "frames_in_flight": n_fif,
            "single_frame": None if single is None else {
                "note": "the same steps, one blocking run_inference_pipeline call per step (frame latency mode)",
                "ms_per_step": single[0] / args.steps, "value": hyp_per_step / (single[0] / args.steps / 1000.0),
                "e2e_value": hyp_per_step / (single[1] / args.steps / 1000.0), "unit": "hypotheses/s"},
            "clocks": clocks,
            "roofline": {"bound": "tensor",
                         "kernel": "tcgen05 implicit-GEMM convolutions (conv_window / conv_igemm / conv_igemm2): the "
                                   "launches of this rank's coarse forward, summed",
                         "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst,
                         "frac_of_sustained_peak": achieved / sustained, "peak_sustained": sustained,
                         "traffic": traffic,
                         "traffic_source": "profiles/conv_traffic.json (one ncu pass of this workload; a constant, not a "
                                           "measurement of this run)" if traffic is not None else None,
                         "algorithmic_activation_bytes": ALGO_CONV_BYTES_PER_HYP * rows_rank if (h, w) == (240, 320) else None,
                         "peak_source": peak_src, "algorithmic_tflop_per_step": algo_tflop_per_step,
                         "executed_tflop_per_step": conv_fl.value / prof_steps / 1e12,
                         "conv_ms_per_step": conv_ms_per_step, "conv_launches_per_step": conv_n.value / prof_steps,
                         "conv_share_of_step": conv_ms_per_step / ms_per_step,
                         "whole_step_tflops": gflop_per_hyp((h, w)) * hyp_per_step / n_gpus / ms_per_step,
                         "whole_step_frac": gflop_per_hyp((h, w)) * hyp_per_step / n_gpus / ms_per_step / burst},
        }
        if n_gpus == 1 and not args.no_torch_baseline and args.workload == "rgb576":
            del est, ests
            torch.cuda.empty_cache()
            try:
                line["gpu_torch_baseline"] = torch_gpu_baseline(sc, quick=True)
            except Exception as exc:  # noqa: BLE001 -- a side measurement, never a reason to lose the bench line
                line["gpu_torch_baseline"] = {"failed": repr(exc)[:300]}
        if n_gpus == 1 and not args.no_cpu_baseline and args.workload == "rgb576":
            line["cpu_baseline"] = cpu_baseline_subprocess(args)
        if outputs is not None:
            write_outputs(outputs, Path(args.dump_outputs))
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    if a.impl == "reference":
        run_reference_arm(a)
    elif a.impl == "torch-gpu":
        run_torch_gpu_arm(a)
    else:
        run_mpx_arm(a)
