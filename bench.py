#!/usr/bin/env python
"""bench.py -- NID cost-evaluations/s of the Nelder-Mead inner solve, BASELINE.json configs (default: C3, the 5 M-point cloud).

Workload (one "step"): S independent inner Nelder-Mead solves of the reference's calibration
(VisualCameraCalibration::estimate_pose_nelder_mead, src/vlcal/calib/visual_camera_calibration.cpp:70-139) with the
reference's default parameters (<= 256 inner iterations, 16 bins, step 1e-3), each from its own start pose (ground truth
+- 0.5 deg / 2 cm in one of 8 sign patterns):
  --config C3 (default)  Livox-Avia-like 5 M-point cloud + 3840x1920 equirectangular camera     (BASELINE configs[2])
  --config C2            Ouster-OS1-64-like 1 M-point cloud + 1920x1080 plumb_bob camera        (BASELINE configs[1])
  --config C5            pose-grid search: 16 384 candidate poses x 5 M points (pinhole), pose-sharded over the ranks
                         (BASELINE configs[4]; a step scores the whole grid)
Metric: NID cost evaluations per second = evaluations the serial reference would have made (speculatively scored candidates
are reported separately) x bags, per second; `mpoints_per_s` counts every point-pose actually projected + binned.

  value : data resident in HBM (culled cloud + image uploaded, cost object built) -- timed region = the solves.
          One solve = ONE launch of the persistent cooperative kernel (csrc/nid_persistent.cuh).
  e2e   : the same step through the host-buffer C ABI (vlcal_estimate_pose_nelder_mead): upload, GPU view culling,
          cost-object construction, solve, result -- host<->device copies inside the timed region.
  --impl reference : the reference's CPU path on a bounded sample of the same step (config.reference_sample): the oracle
          port (oracle/vlcal_oracle.c, pinned bit-for-bit against the reference's own sources compiled in oracle/_ref),
          serial over points and OpenMP over bags exactly like the reference (visual_camera_calibration.cpp:107);
          `reference_build` times oracle/_ref itself beside it.

N > 1 (torchrun, one rank per GPU): weak scaling over bags -- rank r owns bag r, and the joint objective sum_bags NID
(visual_camera_calibration.cpp:105-110) is formed INSIDE the persistent kernel: the finalizing blocks store their scores
into every peer's cudaIpc-shared mailbox over NVLink and every block of every rank adds the contributions in rank order
(torch.distributed / NCCL only bootstraps the handles and the timing barrier).  --exchange nccl: host loop with one NCCL
all-reduce per Nelder-Mead batch instead (A/B).  C5 shards the pose list instead (one all_gather of the scores).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "nid_cost_evals_per_sec"
UNIT = "evals/s"

CONFIGS = {
    "C2": dict(camera="pinhole_1920x1080", pattern="os1_64", points=1_000_000, config_index=1, solves_per_step=40, ref_iterations=12,
               workload="C2: 1M-pt OS1-64-like cloud + 1920x1080 plumb_bob; a step = 40 estimate_pose_nelder_mead inner solves (<=256 NM iterations, 16 bins) from 8 start poses x 5 scales"),
    "C3": dict(camera="equirect_3840x1920", pattern="avia", points=5_000_000, config_index=2, solves_per_step=8, ref_iterations=4,
               workload="C3: 5M-pt Livox-Avia-like non-repetitive cloud + 3840x1920 equirectangular; a step = 8 estimate_pose_nelder_mead inner solves (<=256 NM iterations, 16 bins) from 8 start poses"),
    "C5": dict(camera="pinhole_1920x1080", pattern="avia", points=5_000_000, config_index=4, solves_per_step=1, ref_iterations=0,
               workload="C5: pose-grid search, 16384 candidate poses (8x8x8 rotations +-4 deg x 2x4x4 translations +-10 cm) x 5M-pt cloud, 1920x1080 plumb_bob; a step scores the whole grid"),
}
SIGNS = [(1, 1, 1, 1, 1, 1), (-1, 1, 1, 1, -1, 1), (1, -1, 1, -1, 1, 1), (1, 1, -1, 1, 1, -1), (-1, -1, 1, -1, -1, 1), (1, -1, -1, -1, 1, -1), (-1, 1, -1, 1, -1, -1), (-1, -1, -1, -1, -1, -1)]


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C3", choices=sorted(CONFIGS))
    ap.add_argument("--points", type=int, default=0, help="override the cloud size (parity / smoke runs)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--variant", type=int, default=0, help="kernel variant (0 default, 1 exact-fp64 only, 2/3 points per lane, 4 round-1 kernels)")
    ap.add_argument("--solver", default="auto", choices=["auto", "host", "device", "persistent"], help="inner-solve loop (auto = persistent kernel)")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"], help="N>1: in-kernel peer-memory exchange (default) or host loop + NCCL all-reduce per batch")
    ap.add_argument("--ref-iterations", type=int, default=-1, help="NM iterations per reference-arm step (bounded sample); -1 = per-config default")
    ap.add_argument("--grid-poses", type=int, default=16384, help="C5: poses of the grid (16384 = the BASELINE figure)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float64), to compare two builds output for output")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, outputs):
    """DIR/<name>.npy for every array a caller of the timed path receives, as float64.  The inputs are seeded, so two runs
    with the same arguments can be compared file for file.  Past DUMP_LIMIT_BYTES in all, each array keeps a fixed, seeded,
    sorted sample of its rows."""
    outputs = {k: np.asarray(v, dtype=np.float64) for k, v in outputs.items()}
    total = sum(a.nbytes for a in outputs.values())
    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        if total > DUMP_LIMIT_BYTES and a.ndim > 0 and len(a) > 1:
            keep = max(1, int(len(a) * DUMP_LIMIT_BYTES / total))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(directory, f"{name}.npy"), a)


def start_poses(cfg, T_gt, count):
    """`count` start poses: ground truth (+) the C2 perturbation (0.5 deg, 2 cm per axis) in 8 sign patterns, scaled 1.0 .. 0.6."""
    from direct_visual_lidar_calibration_b200 import synthetic as S

    out = []
    for k in range(count):
        s = SIGNS[k % 8]
        scale = 1.0 - 0.1 * ((k // 8) % 5)
        out.append(S.perturb(T_gt, (0.5 * s[0] * scale, 0.5 * s[1] * scale, 0.5 * s[2] * scale), (0.02 * s[3] * scale, 0.02 * s[4] * scale, 0.02 * s[5] * scale)))
    return out


def make_inputs(args, bag_index):
    from direct_visual_lidar_calibration_b200 import synthetic as S

    cfg = CONFIGS[args.config]
    n = args.points or cfg["points"]
    bag = S.make_bag(cfg["camera"], cfg["pattern"], n, config_index=cfg["config_index"], bag_index=bag_index)
    # every rank must use the same start poses: ground truth of the (shared) camera + the perturbations
    bag["starts"] = start_poses(cfg, S.gt_T_camera_lidar(), max(8, cfg["solves_per_step"]))
    bag["T_init"] = bag["starts"][0]
    return bag


def _make_inputs_star(ab):
    return make_inputs(*ab)


def config_dict(args, world, n_points, W, H):
    """Identical in both arms (the driver compares them): what is computed, on what, and the bounded sample the CPU arm times."""
    cfg = CONFIGS[args.config]
    it = cfg["ref_iterations"] if args.ref_iterations < 0 else args.ref_iterations
    if args.config == "C5":
        sample = "CPU arm: CostCalculatorNID::calculate of the first 4 grid poses on the full cloud per step (the grid is 16384 such evaluations)"
    else:
        sample = f"CPU arm: the first {it} Nelder-Mead iterations of ONE inner solve per step (start pose 0), view culling included; serial over points, OpenMP over bags, as the reference"
    return {"workload": cfg["workload"], "points": n_points, "image": f"{W}x{H}", "bags": world, "parallelism": (f"bags{world}" if args.config != "C5" else f"poses{world}") if world > 1 else "single",
            "reference_sample": sample, "l2": "flushed (256 MiB write) between steps; within a solve the culled cloud is re-read every NM iteration by the algorithm itself"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu_index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def committed_ncu(config):
    """Figures that only a profiler capture gives (DRAM traffic, executed instructions), read from the committed summary of
    THIS config's capture (profiles/r02_ncu_<config>.json, written by tools/ncu_summary.py); None if not captured."""
    path = os.path.join(ROOT, "profiles", f"r02_ncu_{config}.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except Exception:
            pass
    return None


def oracle_objects(bag):
    from oracle import oracle as O

    cam = O.create_camera(bag["camera_model"], bag["intrinsics"], bag["distortion"])
    return O, cam


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, rank, world):
    """--impl reference: the CPU path of the reference on a bounded sample of the step (config.reference_sample).  N > 1: the
    joint objective over N bags with the reference's OpenMP loop over bags (one thread per bag), rank 0 alone."""
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    it = cfg["ref_iterations"] if args.ref_iterations < 0 else args.ref_iterations
    if world > 1:  # the N bags of the joint objective, generated in parallel (the 5 M-point clouds take ~40 s each)
        import concurrent.futures as cf

        with cf.ProcessPoolExecutor(max_workers=min(world, max(1, host_threads() // 4))) as ex:
            bags_in = list(ex.map(_make_inputs_star, [(args, b) for b in range(world)]))
    else:
        bags_in = [make_inputs(args, 0)]
    bag = bags_in[0]
    O, cam = oracle_objects(bag)
    cores = min(world, host_threads())
    O.set_bag_threads(cores)
    W, H = bag["width"], bag["height"]
    times, evals = [], 0
    if args.config == "C5":
        from direct_visual_lidar_calibration_b200 import synthetic as S

        poses = S.pose_grid(bag["T_gt"])[:4]
        fov = O.estimate_camera_fov(cam, W, H)
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            for T in poses:
                O.nid_calculate(cam, bag["image"], bag["points"], bag["intensities"], 16, fov, T)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
                evals += len(poses)
        sample_evals = len(poses)
        ref_build = None
    else:
        p = O.default_calib_params()
        p.max_inner_iterations = it
        bags = [(b["image"], b["points"], b["intensities"]) for b in bags_in]
        per_step = 0
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = O.estimate_pose_nelder_mead(cam, bags, bag["T_init"], p)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
                evals += r["num_evaluations"] * world  # one evaluation = one pose x one bag
                per_step = r["num_evaluations"] * world
        sample_evals = per_step
        # the same bounded sample through the reference's OWN visual_camera_calibration.cpp + cost_calculator_nid.cpp
        # (oracle/_ref, compiled against stand-in third-party headers); the port above is the faster of the two
        ref_build = None
        try:
            from oracle import reference as R

            if R.available():
                rcam = R.Camera(bag["camera_model"], bag["intrinsics"], bag["distortion"])
                sys.stdout.flush()
                saved = os.dup(1)
                devnull = os.open(os.devnull, os.O_WRONLY)
                os.dup2(devnull, 1)  # the reference prints "cost:<best>" to stdout (visual_camera_calibration.cpp:115)
                try:
                    t0 = time.perf_counter()
                    R.calibrate_nelder_mead(rcam, bags, bag["T_init"], max_outer_iterations=1, max_inner_iterations=it)
                    dt = time.perf_counter() - t0
                finally:
                    os.dup2(saved, 1)
                    os.close(saved)
                    os.close(devnull)
                ref_build = {"value": per_step / dt, "unit": UNIT, "cores": cores, "ms_per_step": 1e3 * dt,
                             "note": "VisualCameraCalibration::calibrate (1 outer iteration) from the reference's own sources, stand-in Eigen/cv::Mat/GTSAM headers, -O2"}
        except Exception as e:
            ref_build = {"unavailable": repr(e)}
    total = sum(times)
    value = evals / total
    config = config_dict(args, world, bag["points"].shape[0], W, H)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config, "evals_per_step": sample_evals,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": config["reference_sample"], "reference_build": ref_build},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline(bag, points, intens, max_fov, label):
    """The oracle timed on this box's host cores on a bounded sample (about 10-20 s): (i) reference-faithful -- serial over
    points, one thread (the reference only parallelises over bags); (ii) best-effort -- OpenMP over points, all cores."""
    O, cam = oracle_objects(bag)
    T = bag["T_init"]
    t0 = time.perf_counter()
    O.nid_calculate(cam, bag["image"], points, intens, 16, max_fov, T)  # warm + calibrates the sample size
    t_one = time.perf_counter() - t0
    n_faithful = int(max(3, min(40, 10.0 / max(t_one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n_faithful):
        O.nid_calculate(cam, bag["image"], points, intens, 16, max_fov, T)
    t_f = (time.perf_counter() - t0) / n_faithful
    cores = host_threads()
    O.nid_calculate(cam, bag["image"], points, intens, 16, max_fov, T, omp=True)
    n_omp = int(max(5, min(100, 3.0 / max(t_f / max(1, cores // 4), 1e-4))))
    t0 = time.perf_counter()
    for _ in range(n_omp):
        O.nid_calculate(cam, bag["image"], points, intens, 16, max_fov, T, omp=True)
    t_o = (time.perf_counter() - t0) / n_omp
    n = points.shape[0]
    ref_build = None
    try:  # the reference's own cost_calculator_nid.cpp (oracle/_ref, built where /root/reference exists), same sample
        from oracle import reference as R

        if R.available():
            rcam = R.Camera(bag["camera_model"], bag["intrinsics"], bag["distortion"])
            Ts = [T] * max(2, n_faithful // 4)
            R.nid_calculate(rcam, bag["image"], points, intens, 16, Ts[:1])
            t0 = time.perf_counter()
            R.nid_calculate(rcam, bag["image"], points, intens, 16, Ts)
            t_r = (time.perf_counter() - t0) / len(Ts)
            ref_build = {"value": 1.0 / t_r, "unit": UNIT, "cores": 1, "ms_per_eval": 1e3 * t_r,
                         "note": "CostCalculatorNID::calculate from the reference's own source, compiled against the stand-in Eigen/cv::Mat headers of oracle/ref_standin (-O2, no -march); one thread per bag as in the reference"}
    except Exception as e:  # a missing prebuilt library only removes this cross-check
        ref_build = {"unavailable": repr(e)}
    return {
        "value": 1.0 / t_f, "unit": UNIT, "cores": 1, "kind": "port", "reference_build": ref_build,
        "sample": f"{n_faithful} evaluations of CostCalculatorNID::calculate on {label} ({n} points), serial over points as in the reference",
        "ms_per_eval": 1e3 * t_f, "mpoints_per_s": n / t_f * 1e-6,
        "best_effort": {"value": 1.0 / t_o, "unit": UNIT, "cores": cores, "note": "OpenMP over points with thread-private histograms -- NOT what the reference does", "ms_per_eval": 1e3 * t_o},
    }


def rank_cpus(ordered, siblings_of, local_rank, world):
    """CPUs of one rank: the allowed CPUs in NUMA order are grouped into physical cores (a core = its hardware threads),
    the cores are dealt out in equal contiguous runs.  Returns (sorted CPU list, physical cores per rank)."""
    allowed = set(ordered)
    cores, seen = [], set()
    for c in ordered:
        if c in seen:
            continue
        sib = [x for x in siblings_of(c) if x in allowed] or [c]
        cores.append(sib)
        seen.update(sib)
    per = len(cores) // world
    if per < 1:
        return [], 0
    return sorted(x for core in cores[local_rank * per : (local_rank + 1) * per] for x in core), per


def bind_rank_to_cores(local_rank, world):
    """One slice of the host's cores per rank, NUMA node by NUMA node, whole physical cores (what `numactl` does for a
    launcher): the e2e path converts and uploads 200 MB of host doubles per solve at C3, and with every rank's pages and
    conversion threads on whichever node the scheduler picked, two ranks ran that at 2.7x the single-rank time
    (profiles/r02_bench_e_c3_n2.json; 1.2x with the binding, r02_bench_k_c3_n2.json).
    Returns a description for the JSON line (None when nothing was changed)."""
    if world <= 1 or not hasattr(os, "sched_setaffinity"):
        return None
    try:
        import glob

        def cpulist(text):
            out = []
            for part in text.strip().split(","):
                if not part:
                    continue
                a, _, b = part.partition("-")
                out.extend(range(int(a), int(b or a) + 1))
            return out

        allowed = set(os.sched_getaffinity(0))
        nodes = sorted(glob.glob("/sys/devices/system/node/node[0-9]*"), key=lambda d: int(d.rsplit("node", 1)[1]))
        ordered = []
        for d in nodes:
            with open(os.path.join(d, "cpulist")) as f:
                ordered.extend(c for c in cpulist(f.read()) if c in allowed)
        if len(ordered) != len(allowed):
            ordered = sorted(allowed)

        def siblings_of(c):
            try:
                with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                    return cpulist(f.read())
            except OSError:
                return [c]

        mine, per = rank_cpus(ordered, siblings_of, local_rank, world)
        if len(mine) < 2:
            return None
        os.sched_setaffinity(0, mine)
        return {"physical_cores_per_rank": per, "threads_per_rank": len(mine), "numa_nodes": len(nodes), "first_cpu": mine[0], "last_cpu": mine[-1]}
    except Exception as e:  # binding is an optimisation: never fail the run over it
        print(f"[bench] core binding skipped: {e}", file=sys.stderr)
        return None


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    affinity = bind_rank_to_cores(local_rank, world)  # before any buffer is allocated or thread started
    if args.warmup < 3:
        args.warmup = 3
    cfg = CONFIGS[args.config]

    import torch
    import torch.distributed as dist

    import direct_visual_lidar_calibration_b200 as V
    from direct_visual_lidar_calibration_b200 import calibration as VC
    from direct_visual_lidar_calibration_b200 import synthetic as S

    if not os.path.exists(V.library_path()):
        V.build_library()
    if not torch.cuda.is_available() or V.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = local_rank
    V.set_solver_mode({"auto": 0, "host": 1, "device": 2, "persistent": 3}[args.solver])
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    grid_mode = args.config == "C5"
    bag = make_inputs(args, 0 if grid_mode else rank)  # C5: every rank holds a replica of the cloud, the pose list is sharded
    cam = V.create_camera(bag["camera_model"], bag["intrinsics"], bag["distortion"])
    W, H = bag["width"], bag["height"]
    data = V.VisualLiDARData(bag["image"], bag["points"], bag["intensities"])
    starts = bag["starts"][: cfg["solves_per_step"]]

    # all-reduce of the per-pose partial sums over ranks (NCCL, one small collective per Nelder-Mead batch; A/B path only)
    red_dev = torch.zeros(16, dtype=torch.float64, device="cuda")
    red_host = torch.zeros(16, dtype=torch.float64).pin_memory()
    n_collectives = [0]

    def allreduce(vals):
        k = vals.shape[0]
        red_host[:k] = torch.from_numpy(vals)
        red_dev[:k].copy_(red_host[:k], non_blocking=True)
        dist.all_reduce(red_dev[:k])
        red_host[:k].copy_(red_dev[:k], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        vals[:] = red_host[:k].numpy()
        n_collectives[0] += 1

    px = None
    if world > 1 and args.exchange == "p2p" and not grid_mode:
        # fused path: the kernels exchange the scores over NVLink peer memory
        from direct_visual_lidar_calibration_b200.distributed import PeerExchange

        ok = 1.0
        try:
            px = PeerExchange(device, rank, world)
        except Exception as e:  # no peer access / IPC on this box: every rank must take the same decision
            print(f"[bench] rank {rank}: peer exchange unavailable ({e})", file=sys.stderr)
            px, ok = None, 0.0
        flag = torch.tensor([ok], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() == 1.0:
            px.connect_with_torch()
        else:
            if px is not None:
                px.close()
            px = None
            args.exchange = "nccl"
    ar = allreduce if (world > 1 and px is None and not grid_mode) else None

    # ---- resident setup (outside the timed region) ---------------------------------------------------------------------
    params = V.VisualCameraCalibrationParams()
    if grid_mode:
        cost = V.CostCalculatorNID(cam, data, V.NIDCostParams(16), device=device)
        grid = S.pose_grid(bag["T_gt"])
        if args.grid_poses != len(grid):
            grid = grid[np.linspace(0, len(grid) - 1, args.grid_poses).astype(int)]
        n_resident = data.size()
        res_points, res_intens = data.points, data.intensities
    else:
        cull = V.ViewCulling(cam, (W, H), V.ViewCullingParams(True), device=device)
        idx = cull.cull_indices(data.points, bag["T_init"])
        culled = V.VisualLiDARData(bag["image"], data.points[idx], data.intensities[idx])
        cost = V.CostCalculatorNID(cam, culled, V.NIDCostParams(16), device=device)
        n_resident = culled.size()
        res_points, res_intens = culled.points, culled.intensities
    cost.set_kernel_variant(args.variant)
    cost.reorder_for_pose(bag["T_init"])  # same grouping the e2e path gets from its culling pass
    if px is not None:
        cost.attach_peer_exchange(px)
        px.set_default(True)  # cost objects built inside the e2e call attach it too
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def resident_step():
        if grid_mode:
            from direct_visual_lidar_calibration_b200 import initial_guess as IG

            nid = IG.score_poses(cost, grid, rank, world)
            mine = len(grid[rank::world])
            return {"evals": len(grid) / world, "computed": mine, "batches": (mine + 7) // 8, "result": float(np.nanmin(nid)), "outputs": {"grid_nid": nid}}
        ev = cm = bt = 0
        y = None
        solves = []
        for T0 in starts:
            T, r = VC.estimate_pose_on_costs([cost], T0, params, allreduce=ar)
            ev += r["num_evaluations"]
            cm += r["num_evaluations_computed"]
            bt += r["num_batches"]
            y = r["y"]
            solves.append((T, r))
        # per solve: the estimated T_camera_lidar, the Nelder-Mead minimiser and its cost, and the counts of the serial search
        outputs = {"T_camera_lidar": [T for T, _ in solves], "nm_x": [r["x"] for _, r in solves], "nm_cost": [r["y"] for _, r in solves],
                   "nm_converged": [r["converged"] for _, r in solves], "nm_iterations": [r["num_iterations"] for _, r in solves],
                   "nm_evaluations": [r["num_evaluations"] for _, r in solves]}
        return {"evals": ev, "computed": cm, "batches": bt, "result": y, "iterations": r["num_iterations"], "outputs": outputs}

    def e2e_step():
        if grid_mode:
            c = V.CostCalculatorNID(cam, data, V.NIDCostParams(16), device=device)  # host buffers -> device inside the timed region
            nid = V.score_poses([c], grid[rank::world])
            c.close()
            mine = len(grid[rank::world])
            return {"evals": len(grid) / world, "computed": mine, "stats": None, "result": float(np.nanmin(nid))}
        ev = cm = 0
        stats = []
        for T0 in starts:
            calib = V.VisualCameraCalibration(cam, [data], params, device=device, allreduce=ar)
            _, r = calib.estimate_pose_nelder_mead(T0)
            ev += r["num_evaluations"]
            cm += r["num_evaluations_computed"]
            stats.append(calib.stats)
        return {"evals": ev, "computed": cm, "stats": stats}

    def timed(fn, steps, warmup, profile):
        for _ in range(warmup):
            fn()
        results, ms = [], []
        if profile:
            cost.set_profiling(True)
            cost.reset_profile()
        barrier()
        t_wall0 = time.perf_counter()
        for _ in range(steps):
            flush.fill_(1)  # L2 flush between steps (outside the per-step event pair)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            results.append(fn())
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        barrier()
        wall = time.perf_counter() - t_wall0
        prof = cost.profile() if profile else None
        if profile:
            cost.set_profiling(False)
        total_ms = torch.tensor([sum(ms)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
        return results, float(total_ms.item()), wall, prof

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    res, total_ms, wall, prof = timed(resident_step, args.steps, args.warmup, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res[-1]["outputs"])

    evals_ref = sum(r["evals"] for r in res)      # what the serial reference would evaluate (this rank's bag / pose share)
    evals_cmp = sum(r["computed"] for r in res)   # poses actually scored
    batches = sum(r["batches"] for r in res)
    secs = total_ms * 1e-3
    value = world * evals_ref / secs  # every rank scores its own bag (or its share of the pose list) for every evaluation
    mpoints = world * n_resident * evals_cmp / secs * 1e-6

    # ---- e2e: host buffers in, result out, every step -----------------------------------------------------------------------
    e2e_res, e2e_ms, _, _ = timed(e2e_step, args.steps, 3, profile=False)
    e2e_steps = len(e2e_res)
    e2e_evals = sum(r["evals"] for r in e2e_res)
    e2e_cmp = sum(r["computed"] for r in e2e_res)
    e2e_value = world * e2e_evals / (e2e_ms * 1e-3)
    n_solves = 1 if grid_mode else len(starts)
    h2d = n_solves * (16 * data.size() + W * H) + (128 * len(grid[rank::world]) if grid_mode else 0)  # float4 cloud staging + image per solve (+ the pose list)
    d2h = (8 * (e2e_cmp // e2e_steps)) if grid_mode else n_solves * (2400 + 8)  # scores; per solve: final simplex state + counters (+ evaluation trace, 72 B each, when a callback is set)

    # ---- P = 1 roofline point: one pose per pass over the resident cloud (pose-list mode, 1 pose per pass) ---------------------
    p1 = None
    if True:
        Ts1 = np.stack([bag["starts"][k % len(bag["starts"])] for k in range(24)])
        had_px = px is not None
        if had_px:
            cost.attach_peer_exchange(None)  # single-pose roofline point is a per-GPU figure
        cost.set_poses_per_pass(1)
        cost.calculate_batch(Ts1[:4])
        cost.set_profiling(True)
        cost.reset_profile()
        flush.fill_(1)
        torch.cuda.synchronize()
        cost.calculate_batch(Ts1)
        pf1 = cost.profile()
        cost.set_profiling(False)
        cost.set_poses_per_pass(8)
        if had_px:
            cost.attach_peer_exchange(px)
        if pf1["passes"] > 0 and pf1["kernel_ms_total"] > 0:
            p1 = {"us_per_pass": 1e3 * pf1["kernel_ms_total"] / pf1["passes"], "passes": pf1["passes"]}

    if rank != 0:
        if world > 1:
            dist.barrier()
            if px is not None:
                px.close()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (the persistent histogram kernel) ---------------------------------------------------
    peak, peak_src = measured_hbm_peak()
    alg_bytes = 16 * n_resident + W * H  # per PASS over the cloud: float4 points + the image-bin plane (SURVEY 8d), whatever P it carries
    passes = max(1, prof["passes"])
    t_pass = prof["kernel_ms_total"] * 1e-3 / passes
    achieved = alg_bytes / t_pass * 1e-9
    ncu = committed_ncu(args.config)
    poses_per_pass = prof["poses_total"] / passes
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": (ncu or {}).get("dram_bytes_per_pass"), "traffic_source": (ncu or {}).get("source"),
        "peak_source": peak_src, "kernel": "nid_persistent_kernel", "us_per_pass": 1e6 * t_pass, "passes_per_launch": passes / max(1, prof["kernel_launches"]),
        "avg_launch_us": 1e3 * prof["kernel_ms_total"] / max(1, prof["kernel_launches"]), "algorithmic_bytes_per_pass": alg_bytes,
        "poses_per_pass": poses_per_pass, "kernel_share_of_step": prof["kernel_ms_total"] / total_ms,
        "note": "achieved = algorithmic bytes of one pass over the cloud (16 B/point + W*H) / average pass time (launch duration / passes, CUDA events on the launch stream); "
                "a pass carries poses_per_pass poses, i.e. that many times the arithmetic of its byte count, and the cloud is L2-resident across the passes of a solve by design",
    }
    if p1:
        a1 = alg_bytes / (p1["us_per_pass"] * 1e-6) * 1e-9
        roofline["p1"] = {"achieved": a1, "frac": a1 / peak, "us_per_pass": p1["us_per_pass"], "poses_per_pass": 1, "mpoints_per_s": n_resident / p1["us_per_pass"],
                          "note": "same kernel, pose-list mode with one pose per pass (vlcal_nid_set_poses_per_pass): the HBM-bound regime of the path"}
    # the bound that is active at Nelder-Mead batch sizes: instruction issue.  Instructions per point-pose come from the committed
    # ncu capture of this config (not hard-coded); 148 SMs x 4 schedulers x 1 warp-instruction/clk x 32 lanes at the sampled clock.
    sm_clock_hz = 1e6 * (clocks["sm_mhz"] if clocks and clocks.get("sm_mhz") else 1965.0)
    pp_per_s = n_resident * poses_per_pass / t_pass
    ipp = (ncu or {}).get("warp_inst_per_pointpose")
    if ipp:
        alu_peak = 148 * 4 * 32 * sm_clock_hz / ipp
        roofline["issue_bound"] = {"achieved_pointposes_per_s": pp_per_s, "peak_pointposes_per_s": alu_peak, "frac": pp_per_s / alu_peak, "warp_inst_per_pointpose": ipp,
                                   "source": (ncu or {}).get("source")}
    else:
        roofline["issue_bound"] = {"achieved_pointposes_per_s": pp_per_s, "warp_inst_per_pointpose": None, "note": "no committed ncu capture for this config"}

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        cpu = cpu_baseline(bag, res_points, res_intens, cost.max_fov, "the culled cloud" if not grid_mode else "the full cloud")

    host_break = None
    if not grid_mode:
        flat = [s for r in e2e_res for s in r["stats"]]
        host_break = {k: round(float(np.mean([s[k] for s in flat])), 3) for k in ("upload_ms", "cull_ms", "solve_ms")}
    config = config_dict(args, world, data.size(), W, H)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak" if not grid_mode else "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "dtype_note": "geometry decided in f64 semantics: fp32 filter with a rigorous error bound + exact f64 recheck (integer histograms identical to the all-f64 kernel); histogram int32; entropies f64",
        "config": config,
        "run": {"culled_points": n_resident, "exchange": (args.exchange if world > 1 and not grid_mode else None), "kernel_variant": args.variant, "solver": args.solver, "solves_per_step": n_solves, "host_cores_of_rank0": affinity},
        "evals_per_step": evals_ref / args.steps, "evals_computed_per_step": evals_cmp / args.steps, "batches_per_step": batches / args.steps,
        "mpoints_per_s": mpoints, "wall_s_timed_region": wall,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms / e2e_steps, "steps": e2e_steps, "host_breakdown_ms_per_solve": host_break},
        "gpu_launches": int(prof["kernel_launches"]),
        "collectives": n_collectives[0],
        "roofline": roofline,
        "cpu_baseline": cpu,
        "clocks": clocks,
        "result": res[-1].get("result"), "nm_iterations": res[-1].get("iterations"),
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        if px is not None:
            px.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
