#!/usr/bin/env python
"""Benchmark of the AVDN hot path on B200 (contract: see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload train|render|rollout|et_rollout|bert|train_bert|train_rollout|mapprep]
    python bench.py --impl reference ...        # the reference's CPU path, same metric
    python bench.py --dump-outputs DIR ...      # also write the last timed step's outputs as DIR/<name>.npy

One JSON line on stdout (rank 0).  Under torchrun (N>1) every rank runs its shard
of the workload; the timed region is bracketed by a barrier + synchronize and the
maximum over ranks is reported.
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

import numpy as np
import torch


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d["bf16_tflops_sustained"],
                    source="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        while not self._stop.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                    "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in o.strip().split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ===================================================================== render
class RenderWorkload:
    """BASELINE.json configs[2]: 4096 random drone poses, rotated crop + bilinear
    resample from a synthetic 3000x3000 RGB tile to 224x224 views."""

    name = "render_cfg3"
    metric = "rendered views/s"
    unit = "views/s"
    dtype = "u8"
    P_TOTAL = 4096
    SIZE = 3000

    def __init__(self, rank, world):
        from avdn_b200.utils import synthetic as wo   # synthetic inputs (product-side generators)
        self.rank, self.world = rank, world
        self.tile = wo.synthetic_tile(seed=0, size=self.SIZE)
        allc = wo.synthetic_pose_corners(self.P_TOTAL * world, seed=0, size=self.SIZE)
        self.corners = allc[rank * self.P_TOTAL:(rank + 1) * self.P_TOTAL]     # shard by pose
        self.P = self.corners.shape[0]

    def units_per_step(self):
        return self.P

    def config(self):
        return {"workload": "env.py view rendering: 4096 poses/GPU, 3000x3000x3 u8 tile -> 224x224x3 u8 views "
                            "(BASELINE configs[2])",
                "poses_per_gpu": self.P, "tile": [self.SIZE, self.SIZE, 3],
                "cache": "outputs (616 MB/step) exceed L2; the packed tile (72 MB of row-pair records) is L2-resident by design",
                "parallelism": f"pose-sharded x{self.world}, no collective"}

    def setup_gpu(self, dev):
        from avdn_b200.env import ViewRenderer
        self.dev = dev
        self.r = ViewRenderer(dev)
        self.r.add_map("tile", self.tile, None)
        self.corners_dev = torch.from_numpy(self.corners).to(dev)
        self.corners_pin = torch.from_numpy(self.corners).pin_memory()
        self.out = {"views": torch.empty((self.P, 224, 224, 3), dtype=torch.uint8, device=dev)}
        self.host_views = torch.empty((self.P, 224, 224, 3), dtype=torch.uint8).pin_memory()
        self.ev_k = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        self.kernel_ms = []

    def step(self):
        minv = self.r.homography(self.corners_dev)
        self.ev_k[0].record()
        self.r.render(None, None, views=True, minv=minv, out=self.out)
        self.ev_k[1].record()
        return 2                                            # kernels launched

    def after_step(self, timed):
        if timed:
            self.ev_k[1].synchronize()
            self.kernel_ms.append(self.ev_k[0].elapsed_time(self.ev_k[1]))

    def step_e2e(self):
        c = self.corners_pin.to(self.dev, non_blocking=True)
        self.r.render(c, None, views=True, out=self.out)
        self.host_views.copy_(self.out["views"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return int(self.corners_pin.numel() * 4), int(self.host_views.numel())

    def roofline(self, peaks):
        alg = self.P * 224 * 224 * 3 + self.SIZE * self.SIZE * 3
        ms = float(np.mean(self.kernel_ms)) if self.kernel_ms else None
        ach = alg / (ms * 1e-3) / 1e9 if ms else None
        return {"kernel": "render_kernel", "bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
                "frac": (ach / peaks["hbm"]) if ach else None, "traffic": None,
                "peak_source": peaks["source"] + " (burst copy)", "algorithmic_bytes_per_launch": alg,
                "kernel_ms": ms}

    # the reference's own CPU path: cv2 calls of src/env.py:287,290
    def cpu_step(self, n):
        import cv2
        dst = np.array([[0, 0], [223, 0], [223, 223], [0, 223]], dtype=np.float32)
        for c in self.corners[:n]:
            M = cv2.getPerspectiveTransform(c.astype(np.float32), dst)
            cv2.warpPerspective(self.tile, M, (224, 224))
        return n

    def cpu_info(self):
        import cv2
        return {"kind": "reference", "cores": int(cv2.getNumThreads()),
                "what": "cv2.getPerspectiveTransform + cv2.warpPerspective (the calls at src/env.py:287,290)"}

    CPU_SAMPLE = 512


# ================================================================= map preparation
class MapPrepWorkload:
    """SURVEY.md §8f N2 (src/env.py:217-231): per map, INTER_AREA width rescale of the decoded 3000x3000 tile,
    the attention raster (8 filled circles) and the renderer's packed layout, 8 maps per step."""
    name = "mapprep_n2"
    metric = "prepared maps/s"
    unit = "maps/s"
    dtype = "u8"
    MAPS = 8
    SIZE = 3000
    RATIO = (0.7593e-5, 1.0e-5)          # lng_ratio, lat_ratio at ~40 degrees latitude
    CPU_SAMPLE = 8

    def __init__(self, rank, world):
        from avdn_b200.utils import synthetic as syn
        self.rank, self.world = rank, world
        self.tile = syn.synthetic_tile(seed=rank, size=self.SIZE)
        rng = np.random.default_rng(rank)
        self.new_w = int(self.SIZE * self.RATIO[0] / self.RATIO[1])
        self.spots = [((int(rng.integers(0, self.new_w)), int(rng.integers(0, self.SIZE))), int(rng.integers(30, 150)))
                      for _ in range(8)]

    def units_per_step(self):
        return self.MAPS

    def config(self):
        return {"workload": "map preparation (src/env.py:217-231): 3000x3000x3 u8 tile -> INTER_AREA width rescale to "
                            f"{self.new_w} columns + 8 filled attention circles + packed renderer layout, 8 maps per step",
                "maps_per_step": self.MAPS, "tile": [self.SIZE, self.SIZE, 3],
                "cache": "each map moves 27 MB in and ~75 MB out; L2 is flushed between steps",
                "parallelism": f"map-sharded x{self.world}, no collective"}

    def setup_gpu(self, dev):
        from avdn_b200.env import ViewRenderer
        self.dev = dev
        self.r = ViewRenderer(dev)
        self.tile_dev = torch.from_numpy(self.tile).to(dev)
        self.tile_pin = torch.from_numpy(self.tile).pin_memory()
        self.ms = []
        self.ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        self.flag = torch.zeros(1, dtype=torch.int32).pin_memory()

    def _prep(self, tile):
        for i in range(self.MAPS):
            self.r.prepare_map(f"m{i}", tile, self.RATIO[0], self.RATIO[1], self.spots)
        return 4 * self.MAPS

    def step(self):
        self.ev[0].record()
        n = self._prep(self.tile_dev)
        self.ev[1].record()
        return n

    def after_step(self, timed):
        if timed:
            self.ev[1].synchronize()
            self.ms.append(self.ev[0].elapsed_time(self.ev[1]))

    def step_e2e(self):
        h2d = 0
        for i in range(self.MAPS):
            t = self.tile_pin.to(self.dev, non_blocking=True)
            h2d += t.numel()
            self.r.prepare_map(f"m{i}", t, self.RATIO[0], self.RATIO[1], self.spots)
        self.flag.copy_(torch.ones(1, dtype=torch.int32, device=self.dev), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return h2d, 4

    def roofline(self, peaks):
        # algorithmic bytes per map: read the tile once, write the resized tile, write the attention plane, read
        # both and write the 8-byte packed records
        H, W, nw = self.SIZE, self.SIZE, self.new_w
        alg = self.MAPS * (H * W * 3 + H * nw * 3 + H * nw + H * nw * 4 + (H + 1) * (nw + 2) * 8)
        ms = float(np.mean(self.ms)) if self.ms else None
        ach = alg / (ms * 1e-3) / 1e9 if ms else None
        return {"kernel": "resize_area_width_kernel + raster_attention_kernel + pack_tile_kernel", "bound": "hbm",
                "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": (ach / peaks["hbm"]) if ach else None,
                "traffic": None, "peak_source": peaks["source"] + " (burst copy)", "algorithmic_bytes_per_step": alg,
                "step_ms": ms}

    def cpu_step(self, n):
        import cv2
        done = 0
        while done < n:
            im = cv2.resize(self.tile, (self.new_w, self.SIZE), interpolation=cv2.INTER_AREA)
            att = np.zeros((im.shape[0], im.shape[1], 3), np.uint8)
            for c, r in self.spots:
                cv2.circle(att, center=c, radius=r, color=(255, 255, 255), thickness=-1)
            done += 1
        return done

    def cpu_info(self):
        import cv2
        return {"kind": "reference", "cores": int(cv2.getNumThreads()),
                "what": "cv2.resize(INTER_AREA) + np.zeros + cv2.circle (the calls at src/env.py:221-230)"}


WORKLOADS = {"render": RenderWorkload, "mapprep": MapPrepWorkload}
try:
    from bench_train import TrainWorkload, TrainBertWorkload, TrainRolloutWorkload      # noqa: E402
    WORKLOADS["train"] = TrainWorkload
    WORKLOADS["train_bert"] = TrainBertWorkload
    WORKLOADS["train_rollout"] = TrainRolloutWorkload
except ImportError:
    TrainWorkload = None


try:
    from bench_rollout import RolloutWorkload, ETRolloutWorkload      # noqa: E402
    WORKLOADS["rollout"] = RolloutWorkload
    WORKLOADS["et_rollout"] = ETRolloutWorkload
except ImportError:
    RolloutWorkload = None


_RESULT_FD = None


def emit(line):
    """Write the one JSON result line to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    sys.stdout.flush()
    os.write(_RESULT_FD if _RESULT_FD is not None else 1, data)


try:
    from bench_bert import BertWorkload      # noqa: E402
    WORKLOADS["bert"] = BertWorkload
except ImportError:
    BertWorkload = None


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def use_all_host_threads():
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs are meant to use every host core they can."""
    n = os.cpu_count() or 1
    try:
        n = len(os.sched_getaffinity(0))
    except (AttributeError, OSError):
        pass
    if torch.get_num_threads() < n:
        torch.set_num_threads(n)
    try:
        import cv2
        cv2.setNumThreads(n)
    except Exception:
        pass


def run_reference(args, W):
    """``--impl reference``: the reference's CPU implementation of the path (cv2 for the renderer; the oracle port
    pinned to the reference modules for the training step -- the reference tree is not part of this project) on the
    box's host cores, on a bounded sample of the workload.  The line states ITS OWN configuration."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    use_all_host_threads()
    wl = W(0, 1)
    n = wl.CPU_SAMPLE
    for _ in range(args.warmup):
        wl.cpu_step(max(1, n // 8))
    t0 = time.perf_counter()
    units = 0
    for _ in range(args.steps):
        units += wl.cpu_step(n)
    dt = time.perf_counter() - t0
    val = units / dt
    info = wl.cpu_info()
    cfg = dict(wl.config())
    cfg.update(getattr(wl, "cpu_config", lambda: {})())
    cfg["device"] = "cpu"
    cfg["gpu_arm_workload"] = wl.config()["workload"]
    line = {"impl": "reference", "metric": wl.metric, "value": val, "unit": wl.unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": getattr(wl, "cpu_dtype", wl.dtype), "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": val, "unit": wl.unit, "cores": info["cores"], "kind": info["kind"],
                             "sample": f"{n} units per step of the workload, {info['what']}"},
            "e2e": {"value": val, "unit": wl.unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


DUMP_SAMPLE = 1 << 20          # elements kept of a larger output (fixed seeded indices)
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(wl, out_dir):
    """``--dump-outputs``: write the arrays of ``wl.outputs()`` (what the last timed step computed) as
    ``<name>.npy``, float64 where the output is float64 and float32 otherwise.  An output of more than
    ``DUMP_SAMPLE`` elements is reduced to a sample at indices drawn from a generator seeded by its name, so that
    two builds of the project can be compared array for array."""
    import zlib
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in sorted(wl.outputs().items()):
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
            idx = torch.randint(0, t.numel(), (DUMP_SAMPLE,), generator=g).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        a = t.cpu().numpy().astype(np.float64 if t.dtype == torch.float64 else np.float32)
        total += a.nbytes
        if total > DUMP_MAX_BYTES:
            raise RuntimeError(f"--dump-outputs: the outputs exceed {DUMP_MAX_BYTES >> 20} MB at {name}")
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measure(wl, dev, rank, world, local, steps, warmup, with_cpu, dist, dump_dir=None):
    """One workload, the bench contract: W untimed warm-up steps, exactly K timed steps bracketed by barrier +
    synchronize, CUDA events on the launching stream, L2 flushed between timed steps, max over ranks; then the same
    metric end to end through the public API with host buffers; then the roofline of the dominant kernel and (rank 0)
    the CPU leg.  With ``dump_dir`` rank 0 writes the outputs of the last timed step there first (``dump_outputs``).
    Returns the result dict on every rank (the CPU leg and the formatting only matter on rank 0)."""
    use_dist = dist is not None
    peaks = load_peaks()

    def barrier():
        if use_dist:
            dist.barrier()
        torch.cuda.synchronize()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > L2 (126 MB)
    launches = 0
    before_step = getattr(wl, "before_step", lambda: None)
    for _ in range(warmup):
        before_step()
        wl.step()
        wl.after_step(False)
    barrier()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ClockSampler(local) as clk:
        barrier()
        t_wall0 = time.perf_counter()
        for i in range(steps):
            before_step()                                   # untimed
            flush.zero_()                                   # L2 flush between timed iterations (untimed)
            evs[i][0].record()
            launches += wl.step()
            evs[i][1].record()
            wl.after_step(True)
        barrier()
        t_wall = time.perf_counter() - t_wall0
    if dump_dir is not None and rank == 0:
        dump_outputs(wl, dump_dir)
    ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if use_dist:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    units = wl.units_per_step() * world * steps
    value = units / (ms * 1e-3)

    # end-to-end through the public API with host buffers
    for _ in range(2):
        wl.step_e2e()
    barrier()
    e_steps = max(3, min(steps, 10))
    t0 = time.perf_counter()
    for _ in range(e_steps):
        h2d, d2h = wl.step_e2e()
    barrier()
    te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if use_dist:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = wl.units_per_step() * world * e_steps / float(te.item())

    # collective parts of the roofline measurement (the instrumented training step all-reduces) and the
    # multi-GPU proofs run on every rank; only rank 0 formats the result
    prep = getattr(wl, "prepare_roofline", None)
    if prep is not None:
        prep()
    barrier()
    multi = None
    mg = getattr(wl, "multi_gpu_checks", None)
    if mg is not None and use_dist:
        multi = mg(dist)
    barrier()
    del flush
    cpu = None
    if rank == 0 and with_cpu:
        use_all_host_threads()
        n = wl.CPU_SAMPLE
        wl.cpu_step(max(1, n // 8))
        t0 = time.perf_counter()
        done = wl.cpu_step(n)
        dt = time.perf_counter() - t0
        info = wl.cpu_info()
        cpu = {"value": done / dt, "unit": wl.unit, "cores": info["cores"], "kind": info["kind"],
               "sample": f"{n} units of the workload, {info['what']}; {dt:.1f} s of CPU time"}
    line = {"metric": wl.metric, "value": value, "unit": wl.unit, "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms / steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": wl.dtype, "data": "synthetic",
            "config": wl.config(), "roofline": wl.roofline(peaks) if rank == 0 else None, "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": wl.unit, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "clocks": clk.summary(),
            # host time of the whole timed loop: it also counts the untimed L2 flushes and before_step restores
            "wall_s_timed_region": t_wall}
    if multi:
        line.update(multi)
    extra = getattr(wl, "extra", None)
    if extra and rank == 0:
        line.update(extra(ms / steps))
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train" if "train" in WORKLOADS else "render", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="train workload only: skip the render (configs[2]) and rollout (configs[4]) entries")
    ap.add_argument("--no-library-bar", action="store_true",
                    help="train workload only: skip the stock torch / cuDNN / cuBLAS timing of the same step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="training workloads (train, train_bert, train_rollout) only: after the timed steps, write "
                         "what the last one computed as DIR/<name>.npy (float32 / float64, a fixed seeded sample of "
                         "large outputs, 64 MB at most); the inputs are the same from run to run, so two builds can "
                         "be compared output for output.  The secondary entries of the default line are not dumped")
    args = ap.parse_args()
    # stdout carries exactly ONE line (the JSON result): anything libraries print on file descriptor 1
    # (e.g. NCCL's version banner) is sent to stderr instead
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    W = WORKLOADS[args.workload]
    if args.dump_outputs is not None and (args.impl != "ours" or not hasattr(W, "outputs")):
        raise SystemExit(f"--dump-outputs is available for the GPU arm of the workloads "
                         f"{sorted(k for k, w in WORKLOADS.items() if hasattr(w, 'outputs'))}")

    if args.impl == "reference":
        args.warmup = min(args.warmup, 1)
        run_reference(args, W)
        return

    rank, world, local = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    wl = W(rank, world)
    wl.setup_gpu(dev)
    line = measure(wl, dev, rank, world, local, args.steps, args.warmup, not args.no_cpu_baseline, dist,
                   dump_dir=args.dump_outputs)

    if args.workload == "train":
        # BASELINE.json's metric names two more numbers -- "rendered views/s" (configs[2]) and the greedy rollout
        # of configs[4] "at 1 and 8 B200": measured here, in the same run, as `secondary` entries of the one line.
        # Under torchrun every rank renders / rolls out its own shard (pose- / episode-sharded, no collective).
        if not args.no_library_bar and world == 1:
            line["library_bar"] = wl.library_bar(line["ms_per_step"])
        del wl
        torch.cuda.empty_cache()
        if not args.no_secondary:
            sec = {}
            for name, st, wu in (("render", 10, 3), ("rollout", 3, 3)):
                if name not in WORKLOADS:
                    continue
                w2 = WORKLOADS[name](rank, world)
                w2.setup_gpu(dev)
                r = measure(w2, dev, rank, world, local, st, wu, not args.no_cpu_baseline and world == 1, dist)
                sec[name] = {k: r[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
                                               "dtype", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches",
                                               "clocks")}
                del w2
                torch.cuda.empty_cache()
            line["secondary"] = sec
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
