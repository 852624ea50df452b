#!/usr/bin/env python
"""bench.py -- frames/sec of the SE-SSD per-frame hot path on synthetic KITTI-shape clouds.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run, one rank per GPU)
    python bench.py --impl reference ...                      (the reference's CPU path = the oracle port, host cores)
    python bench.py --workload frame-ring|frame-uniform|stress
    python bench.py ... --dump-outputs DIR                    (also write the detections of the last timed step as DIR/<name>.npy)

Workloads (BASELINE.json `configs`; SURVEY.md 8(d) inputs, generators in se-ssd_b200/sessd_data/synth.py):
  frame-ring     configs[1]: car-only inference, batch 1 per launch, full path voxelise -> sparse 3-D encoder -> BEV neck/head ->
                 rotated NMS, seeded "ring-20k" clouds (KITTI-like 64-beam scan).  DEFAULT = the headline line.
  frame-uniform  same path on the "uniform-20k" input (SURVEY 8(d) primary input; over-dilates through the strided convs).
  stress         configs[4] shape on one GPU per rank: "uniform-200k" clouds, batch 16 per launch, max_voxels 200000.
The default line also carries `extra.uniform20k` and `extra.stress` sub-records (N=1 only; --no-extra skips them).

One STEP = `--frames-per-step` frames pushed through `--streams` concurrent engines (one CUDA graph each).
  value : frames/s with the point clouds already resident in HBM (device-side copy selects the frame);
  e2e   : frames/s through FrameEngine.stage()/launch()/results(): host numpy in, pinned H2D and D2H inside the timed region.
Frames are independent => weak scaling: every rank processes its own `frames-per-step` frames per step, no collective.
Weights: seeded random init with a quiet neck + the committed classification calibration (sessd_data/bench_calib.json) -- both arms
load bit-identical parameters; the parity leg matches the CUDA detections to the CPU oracle's BY ANCHOR INDEX.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark writes nothing into the source tree, which may be read-only
for _p in (ROOT, os.path.join(ROOT, "se-ssd_b200"), os.path.join(ROOT, "scripts")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CPU_THREADS = 16          # torch intra-op threads of the CPU oracle arm: FIXED (a probed count made the arm vary 2.7x across boxes)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="frame-ring", choices=["frame-ring", "frame-uniform", "stress"])
    ap.add_argument("--frames-per-step", type=int, default=None, help="default 512 (frame workloads: >= 5 s timed at 20 steps), 16 (stress)")
    ap.add_argument("--streams", type=int, default=None, help="concurrent engines; default 12 (frame workloads), 1 (stress)")
    ap.add_argument("--pool", type=int, default=16, help="distinct synthetic frames per rank")
    ap.add_argument("--cg-deep", type=int, default=None, help="sparse conv pipeline: 1 deep / one CTA per SM, 0 two CTAs per SM (default: the engine's choice)")
    ap.add_argument("--quick", action="store_true", help="skip the e2e / roofline / cpu_baseline / extra legs (tuning runs)")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra.uniform20k / extra.stress sub-records")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the detections computed in the last one as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ------------------------------------------------------------------------------------------------------------------ workloads
WORKLOADS = {
    "frame-ring": dict(cloud="ring", points=20000, batch=1, max_voxels=20000,
                       name="examples/second car-only inference, batch 1, full voxel->sparse3d->BEV->IoU/NMS, synthetic ring-20k clouds"),
    "frame-uniform": dict(cloud="uniform", points=20000, batch=1, max_voxels=20000,
                          name="examples/second car-only inference, batch 1, full voxel->sparse3d->BEV->IoU/NMS, synthetic uniform-20k clouds"),
    "stress": dict(cloud="uniform", points=200000, batch=16, max_voxels=200000,
                   name="dense-scene stress: uniform-200k clouds, 0.05 m voxels, batch 16 per launch, full path"),
}


def make_cloud(wl, seed):
    from sessd_data import synth
    w = WORKLOADS[wl]
    return synth.ring_cloud(seed, w["points"]) if w["cloud"] == "ring" else synth.uniform_cloud(seed + (1000 if wl == "stress" else 0), w["points"])


def workload_config(wl):
    """The `config` object of the JSON line: identical for both arms (it names the workload, not how an arm runs it)."""
    w = WORKLOADS[wl]
    return {"workload": w["name"], "cloud": "%s-%dk" % (w["cloud"], w["points"] // 1000), "batch": w["batch"], "points_per_frame": w["points"],
            "max_voxels": w["max_voxels"],
            "weights": "seeded random init, quiet neck, committed cls calibration (sessd_data/bench_calib.json: ~400 candidates/frame)"}


def bench_weights(wl):
    from sessd_data import weights
    layers, ssfa, head = weights.bench_detector_state(WORKLOADS[wl]["cloud"], 0)
    return layers, ssfa, head, weights.kitti_car_anchors()


def dump_outputs(path, frames):
    """--dump-outputs: `frames` are dicts of FrameEngine.results() (box3d_lidar, scores, label_preds, anchor_index) plus `cloud`, the
    index of the frame's input in the seeded cloud pool.  Writes path/<name>.npy: cloud and num_detections per frame, the detections
    of all frames concatenated in frame order; box3d_lidar / scores in float32, integers in float64 (exact)."""
    out = {"cloud": np.float64([d["cloud"] for d in frames]),
           "num_detections": np.float64([len(d["scores"]) for d in frames]),
           "box3d_lidar": np.concatenate([np.asarray(d["box3d_lidar"], np.float32).reshape(-1, 7) for d in frames]),
           "scores": np.concatenate([np.asarray(d["scores"], np.float32) for d in frames]),
           "label_preds": np.concatenate([np.asarray(d["label_preds"], np.float64) for d in frames]),
           "anchor_index": np.concatenate([np.asarray(d["anchor_index"], np.float64) for d in frames])}
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_min_mhz": float(min(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------ CPU arm
def cpu_frames(wl, clouds, layers, ssfa, head, anchors, n, warm=1):
    """The reference's CPU path (oracle/frame.py) on `n` frames after `warm` warm-up frames.  TEST INFRASTRUCTURE, executed here only
    as the timed CPU baseline / parity checker.  Returns (frames/s, per-frame stage seconds, outputs)."""
    from oracle import frame as oframe
    torch.set_num_threads(min(CPU_THREADS, os.cpu_count() or 1))
    lnp = oframe.layers_to_numpy(layers)
    mv = WORKLOADS[wl]["max_voxels"]
    for i in range(warm):
        oframe.frame_detections(clouds[i % len(clouds)], lnp, ssfa, head, anchors, max_voxels=mv)
    stage, outs = {}, []
    t0 = time.perf_counter()
    for i in range(n):
        outs.append(oframe.frame_detections(clouds[i % len(clouds)], lnp, ssfa, head, anchors, max_voxels=mv, timings=stage))
    dt = time.perf_counter() - t0
    return n / dt, {k: round(v / n, 3) for k, v in stage.items()}, outs


def run_reference(args):
    """--impl reference: the CPU path timed on the box's host cores; each step = ONE frame (warm-up bounded in time).  Imports only oracle/ and
    the library-free sessd_data generators: libsessd_b200.so is NOT loaded in this arm."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = args.workload
    layers, ssfa, head, anchors = bench_weights(wl)
    clouds = [make_cloud(wl, s) for s in range(min(args.pool, 4))]
    from oracle import frame as oframe
    torch.set_num_threads(min(CPU_THREADS, os.cpu_count() or 1))
    lnp = oframe.layers_to_numpy(layers)
    mv = WORKLOADS[wl]["max_voxels"]
    budget_s = 150.0
    t0 = time.perf_counter()
    oframe.frame_detections(clouds[0], lnp, ssfa, head, anchors, max_voxels=mv)          # first frame: page-in, thread pools
    t_first = time.perf_counter() - t0
    warm = max(0, min(args.warmup - 1, int(0.25 * budget_s / max(t_first, 1e-3))))
    for i in range(warm):
        oframe.frame_detections(clouds[(i + 1) % len(clouds)], lnp, ssfa, head, anchors, max_voxels=mv)
    steps = args.steps
    stage = {}
    t0 = time.perf_counter()
    for i in range(steps):
        last = oframe.frame_detections(clouds[i % len(clouds)], lnp, ssfa, head, anchors, max_voxels=mv, timings=stage)
    dt = time.perf_counter() - t0
    fps = steps / dt
    if args.dump_outputs:
        boxes, scores, labels, aux = last
        dump_outputs(args.dump_outputs, [dict(box3d_lidar=boxes, scores=scores, label_preds=labels, anchor_index=aux["final_anchor"],
                                              cloud=(steps - 1) % len(clouds))])
    line = {"impl": "reference", "metric": "frames_per_sec", "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "timed_steps": steps, "timed_warmup": 1 + warm, "ms_per_step": 1000.0 * dt / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(wl),
            "run": {"frames_per_step": 1, "note": "CPU oracle port of the reference path, rank 0 only"},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": min(CPU_THREADS, os.cpu_count() or 1),
                             "host_threads_available": os.cpu_count() or 1, "kind": "port",
                             "sample": "%d frames timed (1 frame per step), %d warm-up; per-frame stage seconds %s; the sparse "
                                       "encoder has no CPU implementation in the reference (spconv is GPU/third-party): numpy restatement" % (
                                           steps, 1 + warm, {k: round(v / steps, 3) for k, v in stage.items()})},
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------------ CUDA arm
class Rig:
    """`streams` engines of one workload + a device-resident pool of clouds, with the two timed loops."""

    def __init__(self, wl, streams, pool, rank, world, dev):
        from sessd_b200 import _lib
        from sessd_b200.engine import FrameEngine
        self.wl, self.dev, self.world = wl, dev, world
        w = WORKLOADS[wl]
        self.B = w["batch"]
        self.layers, self.ssfa, self.head, self.anchors = bench_weights(wl)
        # frame f of the global stream belongs to rank f mod world (shard.frames_for_rank); each rank draws its own pool
        self.clouds = [make_cloud(wl, rank + world * j) for j in range(pool)]
        maxpts = max(c.shape[0] for c in self.clouds)
        kw = dict(max_voxels=w["max_voxels"])
        if wl == "stress":
            kw["growth"] = (1.0, 8.0, 8.0, 8.0, 8.0)
        self.engines = []
        for _ in range(streams):
            e = FrameEngine(batch=self.B, max_points_per_frame=maxpts, device=dev, **kw)
            e.load_weights(self.layers, self.ssfa, self.head, self.anchors)
            self.engines.append(e)
        self.pool = torch.zeros((pool, maxpts, 4), dtype=torch.float32, device=dev)
        self.npts = [c.shape[0] for c in self.clouds]
        for j, c in enumerate(self.clouds):
            self.pool[j, : c.shape[0]] = torch.from_numpy(c).to(dev)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        for e in self.engines:
            e.capture()
        self.launches_per_batch = (_lib.launch_count() - l0) // (2 * streams)     # capture() runs the body twice (eager warm-up + capture)
        for e in self.engines:
            e.capture_device_only()
        torch.cuda.synchronize()
        self.main = torch.cuda.current_stream()
        self.h2d = self.d2h = 0

    def timed(self, loop_fn, steps):
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(self.main)
        for e in self.engines:
            e.stream.wait_event(ev0)
        for s in range(steps):
            loop_fn(s)
        for e in self.engines:
            done = torch.cuda.Event()
            done.record(e.stream)
            self.main.wait_event(done)
        ev1.record(self.main)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1)
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def batch_ids(self, s, i, F):
        """pool indices of the B frames of launch i of step s"""
        base = (s * F + i * self.B)
        return [(base + f) % len(self.clouds) for f in range(self.B)]

    def step_device(self, F):
        S, B = len(self.engines), self.B

        def fn(s):
            for i in range(F // B):
                e = self.engines[i % S]
                with torch.cuda.stream(e.stream):
                    off = 0
                    for f, j in enumerate(self.batch_ids(s, i, F)):
                        n = self.npts[j]
                        e.d_points[off:off + n].copy_(self.pool[j, :n], non_blocking=True)
                        off += n
                    e.graph_dev.replay()
        return fn

    def last_step_outputs(self, s, F):
        """What the engines still hold after step s of step_device(F): the detections of every engine's last launch in that step, in
        launch order (a fixed subset of the step's frames), unpacked by FrameEngine.results()."""
        S, frames = len(self.engines), []
        for i in range(max(0, F // self.B - S), F // self.B):
            e = self.engines[i % S]
            e.h_result.copy_(e.d_result)
            e.h_meta.copy_(e.d_meta)
            frames += [dict(d, cloud=j) for j, d in zip(self.batch_ids(s, i, F), e.results())]
        return frames

    def prime_offsets(self):
        """frame offsets of the device-resident loop (all pool clouds have the same point count in these workloads)"""
        for e in self.engines:
            ho = e.h_off.numpy()
            for f in range(self.B + 1):
                ho[f] = f * self.npts[0]
            e.d_off.copy_(e.h_off)
        assert len(set(self.npts)) == 1
        torch.cuda.synchronize()

    def step_host(self, F):
        S, B = len(self.engines), self.B

        def fn(s):
            pending = [False] * S
            for i in range(F // B):
                k = i % S
                e = self.engines[k]
                if pending[k]:
                    e.results()
                n = e.stage([self.clouds[j] for j in self.batch_ids(s, i, F)])
                e.launch()
                pending[k] = True
                self.h2d += n * 16 + e.h_off.numel() * 4
                self.d2h += e.h_result.numel() * 4 + e.h_meta.numel() * 4
            for k in range(S):
                if pending[k]:
                    self.engines[k].results()
        return fn


def run_ours(args):
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = args.workload
    B = WORKLOADS[wl]["batch"]
    S = args.streams or (1 if wl == "stress" else 12)
    F = args.frames_per_step or (16 if wl == "stress" else 512)
    F = max(B, F // B * B)
    if args.cg_deep is not None:
        from sessd_b200 import ops as _ops
        _ops.set_sp_cg_deep(args.cg_deep)
    rig = Rig(wl, S, args.pool, rank, world, dev)
    rig.prime_offsets()

    # ---- value: inputs resident in HBM ---------------------------------------------------------------------------
    fn = rig.step_device(F)
    rig.timed(fn, args.warmup)
    sampler = ClockSampler(local)
    sampler.start()
    ms_value = rig.timed(fn, args.steps)
    clocks = sampler.stop()
    value = world * F * args.steps / (ms_value / 1000.0)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, rig.last_step_outputs(args.steps - 1, F))

    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "workload": wl, "value": value, "streams": S, "frames_per_step": F,
                              "ms_per_frame": ms_value / args.steps / F, "clocks": clocks}))
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    # ---- e2e: host buffers through the public engine API -----------------------------------------------------------
    fn = rig.step_host(F)
    rig.timed(fn, args.warmup)
    rig.h2d = rig.d2h = 0
    ms_e2e = rig.timed(fn, args.steps)
    e2e = world * F * args.steps / (ms_e2e / 1000.0)

    # ---- single-batch latency through the public API (one engine, one batch in flight): host numpy in -> detections out ----------
    lat = []
    e = rig.engines[0]
    for i in range(30):
        t0 = time.perf_counter()
        e.stage([rig.clouds[j] for j in rig.batch_ids(0, i, F)])
        e.launch()
        e.results()
        lat.append((time.perf_counter() - t0) * 1000.0)
    latency = {"median_ms": float(np.median(lat[5:])), "p90_ms": float(np.percentile(lat[5:], 90)),
               "what": "stage() + graph replay (H2D, %d kernels, D2H) + results() of ONE batch of %d frame(s), nothing else in flight; host wall clock" % (
                   rig.launches_per_batch, B)}

    line = None
    if rank == 0:
        peaks = load_peaks()
        roof = dominant_kernel_roofline(rig.engines[0], peaks)
        stages = stage_breakdown(rig.engines[0], [rig.clouds[j] for j in rig.batch_ids(0, 0, F)])
        line = {"metric": "frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_value / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": workload_config(wl),
                "run": {"frames_per_step_per_gpu": F, "streams": S, "parallelism": "frame-sharded x%d, no collective" % world,
                        "timed_region_s": {"value": ms_value / 1000.0, "e2e": ms_e2e / 1000.0},
                        "l2": "no explicit flush: per-frame activation working set (~0.4 GB) exceeds the 126 MB L2; inputs rotate over %d clouds" % args.pool},
                "e2e": {"value": e2e, "unit": "frames/s", "ms_per_step": ms_e2e / args.steps,
                        "h2d_bytes_per_step": rig.h2d // args.steps, "d2h_bytes_per_step": rig.d2h // args.steps},
                "gpu_launches": int(rig.launches_per_batch) * (F // B) * args.steps,
                "launches_per_batch": int(rig.launches_per_batch),
                "clocks": clocks, "roofline": roof, "stages_ms": stages, "latency_single_batch": latency}
        if world == 1:
            n_cpu = 1 if wl == "stress" else 4
            fps, stage, outs = cpu_frames(wl, rig.clouds, rig.layers, rig.ssfa, rig.head, rig.anchors, n_cpu, warm=0 if wl == "stress" else 1)
            line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": min(CPU_THREADS, os.cpu_count() or 1),
                                    "host_threads_available": os.cpu_count() or 1, "kind": "port",
                                    "sample": "%d frames of the same workload after a warm-up frame; per-frame stage seconds %s (sparse encoder: numpy "
                                              "restatement, no CPU implementation exists in the reference)" % (n_cpu, stage)}
            line["parity_vs_oracle"] = parity_vs_oracle(rig, outs)
            if not args.no_extra and wl == "frame-ring":
                # release the headline rig before building the next ones (stress needs ~90 GB)
                del rig
                torch.cuda.empty_cache()
                line["extra"] = {"uniform20k": extra_uniform(args, dev), "stress": extra_stress(args, dev, peaks)}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return {"hbm": float(p["hbm_gbs"]), "tf_burst": float(p["bf16_tflops"]), "tf_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "MEASURED_PEAKS.json (of measured)"}
    except Exception:
        return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "B200_PROFILING.md fallback (of fallback)"}


# ------------------------------------------------------------------------------------------------------------------ parity leg
def match_detections(got, ref_boxes, ref_scores, ref_anchor):
    """Match the CUDA path's detections to the oracle's by anchor index.  Returns a dict with the matched differences and the
    unmatched detections of either side (with their scores: a borderline candidate has a score within rounding of the threshold)."""
    ga = np.asarray(got["anchor_index"], np.int64)
    ra = np.asarray(ref_anchor, np.int64)
    common, gi, ri = np.intersect1d(ga, ra, return_indices=True)
    out = {"n_gpu": int(len(ga)), "n_oracle": int(len(ra)), "n_matched": int(len(common))}
    if len(common):
        db = np.abs(got["box3d_lidar"][gi] - ref_boxes[ri])
        scale = np.maximum(np.abs(ref_boxes[ri]), 1.0)
        out["max_abs_box_diff"] = float(db.max())
        out["max_rel_box_diff"] = float((db / scale).max())
        out["max_abs_score_diff"] = float(np.abs(got["scores"][gi] - ref_scores[ri]).max())
        out["max_rel_score_diff"] = float((np.abs(got["scores"][gi] - ref_scores[ri]) / np.maximum(ref_scores[ri], 1e-12)).max())
        out["same_order"] = bool(np.array_equal(ga[np.sort(gi)], ra[np.sort(ri)]))
    only_g = np.setdiff1d(ga, ra)
    only_r = np.setdiff1d(ra, ga)
    out["unmatched"] = ([{"side": "gpu", "anchor": int(a), "score": float(got["scores"][list(ga).index(a)])} for a in only_g] +
                        [{"side": "oracle", "anchor": int(a), "score": float(ref_scores[list(ra).index(a)])} for a in only_r])
    return out


def parity_vs_oracle(rig, outs):
    """The "IoU vs ref" half of BASELINE.json's metric: FrameEngine detections vs the CPU oracle of the reference path on the same
    frames and the same (bit-identical) weights, matched by anchor index.  Fails loudly when the workload is tie-degenerate."""
    from oracle import cpu as ocpu
    e = rig.engines[0]
    frames, n_m, n_g, n_o = [], 0, 0, 0
    worst = {"max_abs_box_diff": 0.0, "max_rel_box_diff": 0.0, "max_abs_score_diff": 0.0, "max_rel_score_diff": 0.0}
    ious, min_gap, unmatched = [], None, []
    for i, o in enumerate(outs):
        got = e.infer([rig.clouds[(i + f) % len(rig.clouds)] for f in range(rig.B)])[0]      # frame 0 of the batch = cloud i
        ob, osc, aux = o[0].numpy(), o[1].numpy(), o[3]
        m = match_detections(got, ob, osc, aux["final_anchor"].numpy())
        # tie check on BOTH sides: kept scores pairwise distinct (gap > 1e-6 relative), else the kept set depends on tie-breaking
        for sc in (got["scores"], osc):
            if len(sc) > 1:
                s = np.sort(sc.astype(np.float64))
                gap = float(np.min(np.diff(s) / np.maximum(s[1:], 1e-12)))
                min_gap = gap if min_gap is None else min(min_gap, gap)
        n_m += m["n_matched"]; n_g += m["n_gpu"]; n_o += m["n_oracle"]
        for k in worst:
            worst[k] = max(worst[k], m.get(k, 0.0))
        unmatched += [dict(u, frame=i) for u in m["unmatched"]]
        if m["n_matched"]:
            ga, ra = got["anchor_index"], aux["final_anchor"].numpy()
            common, gi, ri = np.intersect1d(ga, ra, return_indices=True)
            iou = ocpu.boxes_iou_bev(ocpu.boxes3d_to_bev(got["box3d_lidar"][gi]), ocpu.boxes3d_to_bev(ob[ri]))
            ious.extend(np.diag(iou).tolist())
        frames.append({k: m[k] for k in ("n_gpu", "n_oracle", "n_matched")})
    if min_gap is not None and min_gap <= 1e-6:
        raise RuntimeError("bench workload is tie-degenerate: two kept detections have scores within 1e-6 (relative) of each other")
    ok = (n_m == n_g == n_o) and worst["max_rel_box_diff"] <= 1e-4 and worst["max_rel_score_diff"] <= 1e-4
    res = {"frames": len(outs), "per_frame": frames, "detections_gpu": n_g, "detections_oracle": n_o, "matched_by_anchor": n_m,
           "matched_fraction": (n_m / max(n_g, n_o, 1)), "unmatched": unmatched[:20], "min_rel_score_gap_between_kept": min_gap,
           "mean_bev_iou_vs_oracle": float(np.mean(ious)) if ious else None, "min_bev_iou_vs_oracle": float(np.min(ious)) if ious else None,
           "tolerance": "boxes and scores <= 1e-4 relative (BASELINE.json north_star); keep sets identical", "pass": bool(ok),
           "what": "FrameEngine detections vs the CPU oracle of the reference path, same frames, bit-identical weights, matched by anchor index"}
    res.update(worst)
    return res


# ------------------------------------------------------------------------------------------------------------------ roofline leg
def read_ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the kernel from the newest committed profiles/r2*_ncu.txt summary
    (written by scripts/ncu_summary.py from an `ncu --set full` capture); None when no capture of this round names the kernel."""
    import glob
    import re
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r2*_ncu.txt"))):
        try:
            txt = open(path).read()
        except OSError:
            continue
        for block in txt.split("== ")[1:]:
            if kernel_substr not in block.splitlines()[0]:
                continue
            rd = re.search(r"dram__bytes_read\.sum\s+([0-9.]+) (\w+)", block)
            wr = re.search(r"dram__bytes_write\.sum\s+([0-9.]+) (\w+)", block)
            if rd and wr:
                unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
                best = (float(rd.group(1)) * unit.get(rd.group(2), 1.0) + float(wr.group(1)) * unit.get(wr.group(2), 1.0),
                        os.path.relpath(path, ROOT))
                break
    return best


def dominant_kernel_roofline(e, peaks, reps=20):
    """The conv3x3 128->128 @200x176 layer (largest share of the step; 5 of the 13 neck launches have this shape), timed alone with
    CUDA events on the engine stream, through the same runner call the frame graph uses, L2 flushed before every launch.
    Two-term fp16 split: THREE kind::f16 products per algorithmic MAC (fp32-level parity) => ceiling of `frac` against the bf16 peak is 1/3."""
    neck = e.neck
    flops = 2.0 * neck.batch * neck.h * neck.w * 128 * 128 * 9
    flush = torch.empty((64 * 1024 * 1024,), dtype=torch.float32, device=e.device)   # 256 MB > L2
    launch, kern = neck.bench_layer("bottom_up_block_0.4")
    ms = []
    with torch.cuda.stream(e.stream):
        for _ in range(3):
            launch()
        for _ in range(reps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(e.stream)
            launch()
            b.record(e.stream)
            e.stream.synchronize()
            ms.append(a.elapsed_time(b))
    t = float(np.mean(ms)) / 1000.0
    tr = read_ncu_traffic(kern.split(" ")[0])
    return {"kernel": kern + ", conv3x3 128->128 @200x176 x batch %d" % neck.batch, "bound": "tensor", "achieved": flops / t / 1e12,
            "unit": "TFLOP/s", "peak": peaks["tf_burst"], "peak_source": peaks["source"] + ", bf16 burst (kernel timed alone)",
            "frac": flops / t / 1e12 / peaks["tf_burst"], "avg_launch_ms": t * 1000.0, "algorithmic_flops": flops,
            "traffic": tr[0] if tr else None, "traffic_unit": "bytes/launch (ncu dram read + write)", "traffic_source": tr[1] if tr else None,
            "tensor_work_factor": 3,
            "timing": "CUDA events on the launch stream, L2 flushed (256 MB memset) before every launch, mean of %d" % reps}


def stage_breakdown(e, clouds):
    """Eager single-batch per-stage device times (informational)."""
    from sessd_b200 import ops
    e.stage(clouds)
    out = {}
    with torch.cuda.stream(e.stream):
        e.d_points.copy_(e.h_points, non_blocking=True)
        e.d_off.copy_(e.h_off, non_blocking=True)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record(e.stream)
        ops.voxelize(e.d_points, e.d_off, e.vox)
        ev[1].record(e.stream)
        head = e.sparse_and_neck(mark=lambda label: ev[2].record(e.stream) if label == "dense" else None)
        ev[3].record(e.stream)
        ops.postprocess(head, e.anchors, None, e.post)
        ev[4].record(e.stream)
        e.stream.synchronize()
    for k, name in enumerate(("voxelize", "sparse_encoder", "neck_head", "postprocess")):
        out[name] = round(ev[k].elapsed_time(ev[k + 1]), 4)
    return out


# ------------------------------------------------------------------------------------------------------------------ extra sub-records
def extra_uniform(args, dev):
    """frame-uniform (SURVEY 8(d) primary input) through the same loops, shorter: value, e2e and parity."""
    wl, F, S = "frame-uniform", 192, 12
    rig = Rig(wl, S, 8, 0, 1, dev)
    rig.prime_offsets()
    fn = rig.step_device(F)
    rig.timed(fn, 3)
    ms = rig.timed(fn, 8)
    fn = rig.step_host(F)
    rig.timed(fn, 2)
    ms_h = rig.timed(fn, 8)
    fps, stage, outs = cpu_frames(wl, rig.clouds, rig.layers, rig.ssfa, rig.head, rig.anchors, 2)
    rec = {"config": workload_config(wl), "value": F * 8 / (ms / 1000.0), "e2e": F * 8 / (ms_h / 1000.0), "unit": "frames/s",
           "steps": 8, "frames_per_step": F, "streams": S, "cpu_baseline": {"value": fps, "cores": min(CPU_THREADS, os.cpu_count() or 1), "stage_s": stage},
           "parity_vs_oracle": parity_vs_oracle(rig, outs)}
    del rig
    torch.cuda.empty_cache()
    return rec


def extra_stress(args, dev, peaks):
    """BASELINE configs[4] shape on this GPU: throughput through one batch-16 engine + the per-launch-group roofline fractions of the
    kernels north_star names (sparse-conv GEMM: tensor; rulebook / voxelise / dense scatter: HBM), from scripts/kernel_rooflines.py."""
    import kernel_rooflines as kr
    wl = "stress"
    rig = Rig(wl, 1, 16, 0, 1, dev)
    rig.prime_offsets()
    F = 16
    fn = rig.step_device(F)
    rig.timed(fn, 2)
    ms = rig.timed(fn, 5)
    fn = rig.step_host(F)
    rig.timed(fn, 1)
    ms_h = rig.timed(fn, 5)
    groups = kr.group_rooflines(rig.engines[0], rig.clouds[:16], iters=3)
    keep = [g for g in groups["groups"] if g["group"].startswith(("voxelize", "hash", "rulebook", "conv:", "split", "dense"))]
    tensor = [g for g in keep if g.get("bound") == "tensor" and g.get("impl") not in ("rows",)]
    hbm = [g for g in keep if g.get("bound") == "hbm"]
    rec = {"config": workload_config(wl), "value": F * 5 / (ms / 1000.0), "e2e": F * 5 / (ms_h / 1000.0), "unit": "frames/s", "steps": 5,
           "frames_per_step": F, "ms_per_batch_graph": ms / 5, "eager_total_ms": groups["total_ms"], "voxels": groups["voxels"],
           "active_sites": groups["active_sites"], "peaks": groups["peaks"],
           "sparse_gemm_frac_of_bf16_sustained": {g["group"]: g["frac_bf16"] for g in tensor},
           "hbm_kernel_frac_of_hbm_peak": {g["group"]: g["frac"] for g in hbm},
           "groups": keep, "note": groups["note"]}
    del rig
    torch.cuda.empty_cache()
    return rec


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
