#!/usr/bin/env python
"""Benchmark of the iSDF training hot path (BASELINE.json metric: SDF-MLP train iters/sec and
ray-samples/sec).  One "step" = one Trainer.step(): K1 sampling -> K4 fused PE+MLP forward /
input-gradient / losses / double back-prop -> K5 -> [C1 all-reduce] -> K6 AdamW+re-pack.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision bf16x3|bf16|fp32]
                  [--workload default|scannet|c4|c5] [--dump-outputs DIR]

Prints ONE JSON line (contract in the task statement): metric/value/unit (device-resident inputs),
e2e (public API with host frames, H2D + D2H inside the timed region), roofline (dominant kernel,
CUDA-event timed inside the library), cpu_baseline (oracle port on the host cores), clocks.
`--impl reference` times the CPU port of the reference's own step instead (rank 0 only).
`--dump-outputs DIR` writes what the timed step path computes as DIR/<name>.npy (float32, at most 64 MB); the inputs are
seeded, so two builds run with the same arguments can be compared output for output."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[1]: replicaCAD default config, 1200x680, 200 rays/frame x 5 frames x 27 samples
    "default": dict(H=680, W=1200, fx=600.0, fy=600.0, cx=599.5, cy=339.5, n_rays=200, n_strat=19, n_surf=8,
                    hidden=256, block=2, keyframes=8, name="replicaCAD-default 1200x680 5x200 rays x 27 samples, 256x(2+2) MLP"),
    # configs[2]: ScanNet shapes
    "scannet": dict(H=480, W=640, fx=577.87, fy=577.87, cx=319.5, cy=239.5, n_rays=200, n_strat=19, n_surf=8,
                    hidden=256, block=2, keyframes=8, name="ScanNet-shape 640x480 5x200 rays x 27 samples"),
    # configs[3]: synthetic 640x480, 4096 rays/frame x 64 samples
    "c4": dict(H=480, W=640, fx=577.87, fy=577.87, cx=319.5, cy=239.5, n_rays=4096, n_strat=56, n_surf=8,
               hidden=256, block=2, keyframes=8, name="synthetic 640x480 5x4096 rays x 64 samples"),
    # configs[4]: wide MLP 512x8 (hidden 512, hidden_layers_block 4), 8192 rays/frame x 128 samples.  The tcgen05 kernels
    # take hidden = 256 only: this model runs on the library's fp32 CUDA-core kernels (Trainer falls back with a warning)
    "c5": dict(H=480, W=640, fx=577.87, fy=577.87, cx=319.5, cy=239.5, n_rays=8192, n_strat=120, n_surf=8,
               hidden=512, block=4, keyframes=8, name="wide MLP 512x(4+4), synthetic 640x480 5x8192 rays x 128 samples"),
    # row N1: forward-only evaluation of the grid_dim^3 lattice (Trainer.get_sdf_grid, trainer.py:1426-1444)
    "grid": dict(H=680, W=1200, fx=600.0, fy=600.0, cx=599.5, cy=339.5, n_rays=200, n_strat=19, n_surf=8,
                 hidden=256, block=2, keyframes=1, grid_dim=200,
                 name="get_sdf_grid 200^3 lattice (8.0 M points, forward-only K2, lattice generated in-kernel), 256x(2+2) MLP"),
}
PEAKS_FALLBACK = dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0)
DUMP_MAX_ELEMENTS = 1 << 22          # per array (16 MB of float32); a dump holds at most three arrays this large


def host_copy(t):
    """float32 numpy copy of a device or host tensor; an array above DUMP_MAX_ELEMENTS is cut to a fixed seeded sample
    of its flattened elements (the same positions in every run of the same workload)."""
    import numpy as np
    a = t.detach().float().cpu().numpy().copy()
    if a.size > DUMP_MAX_ELEMENTS:
        idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMENTS, replace=False))
        a = a.reshape(-1)[idx]
    return a


def make_trainer(dev, wl, precision, rank=0, world=1, dist=None):
    """The seeded Trainer of the timed path with this rank's keyframe shard (frames rank, rank + world, ...) resident."""
    import numpy as np
    from isdf.modules import trainer as trainer_mod
    np.random.seed(1 + rank)
    torch.manual_seed(1 + rank)
    tr = trainer_mod.Trainer(dev, make_config(wl, precision, "fast"), incremental=True)
    if dist is not None:                            # identical replicas: broadcast rank 0's parameters
        dist.broadcast(tr.sdf_map.flat_parameters(), 0)
    for i in range(wl["keyframes"]):
        tr.last_is_keyframe = True
        tr.add_data(tr.get_data([rank + i * world]))
    return tr


def reproducible_step(dev, wl, precision, n_steps=3):
    """What the timed step path returns and leaves in the model, from a state every run reproduces: a Trainer seeded and
    loaded like the timed one takes n_steps steps (a new layout's first step runs eagerly, the second captures the CUDA
    graph, the third replays it as every timed step does) and its last step is recorded.  The timed trainer's own last
    step is not reproducible: the library sums gradients and losses with float atomics, so two runs of one build differ in
    the last bits every step, and over hundreds of steps AdamW and the loss-weighted keyframe window grow that into
    visibly different trajectories."""
    tr = make_trainer(dev, wl, precision)
    for _ in range(n_steps):
        losses, _ = tr.step(sync=False)
    torch.cuda.synchronize(dev)
    out = {k: host_copy(v) for k, v in losses.items()}
    out.update(sdf=host_copy(tr.last_sdf), loss_mat=host_copy(tr.last_loss_mat),
               params=host_copy(tr.sdf_map.flat_parameters()), frame_avg_losses=host_copy(tr.frames.frame_avg_losses))
    return out


def write_dump(out_dir, arrays):
    import numpy as np
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured (MEASURED_PEAKS.json)"
        return d
    d = dict(PEAKS_FALLBACK)
    d["_source"] = "fallback (B200_PROFILING.md)"
    return d


def make_config(wl, precision, rng_mode):
    return {
        "dataset": {"format": "synthetic", "depth_scale": 1000.0, "fps": 30, "n_frames": 4000,
                    "camera": {"w": wl["W"], "h": wl["H"], "fx": wl["fx"], "fy": wl["fy"], "cx": wl["cx"], "cy": wl["cy"]}},
        "eval": {"do_vox_comparison": 0, "do_eval": 0, "eval_freq_s": 1, "sdf_eval": 1, "mesh_eval": 0},
        "save": {"save_period": 10, "save_checkpoints": 0, "save_slices": 0, "save_meshes": 0},
        "optimiser": {"lr": 0.0013, "weight_decay": 0.012},
        "trainer": {"steps": 20000},
        "sample": {"n_rays": wl["n_rays"], "n_rays_is_kf": 400, "n_strat_samples": wl["n_strat"],
                   "n_surf_samples": wl["n_surf"], "depth_range": [0.07, 12.0], "dist_behind_surf": 0.1},
        "model": {"refine_poses": 0, "do_active": 0, "frac_time_perception": 1.0, "scale_output": 0.14,
                  "noise_std": 0.25, "noise_kf": 0.08, "noise_frame": 0.04, "window_size": 5,
                  "hidden_layers_block": wl["block"], "hidden_feature_size": wl["hidden"], "iters_per_kf": 60,
                  "iters_per_frame": 10, "kf_dist_th": 0.1, "kf_pixel_ratio": 0.65,
                  "embedding": {"scale_input": 0.05937489, "n_embed_funcs": 5, "gauss_embed": 0,
                                "gauss_embed_std": 11, "optim_embedding": 0}},
        "loss": {"bounds_method": "ray", "loss_type": "L1", "trunc_weight": 5.38344020,
                 "trunc_distance": 0.29365022, "eik_weight": 0.268, "eik_apply_dist": 0.1, "grad_weight": 0.018,
                 "orien_loss": 0},
        "pose_refine": {"pose_lr": 0.0004},
        "b200": {"precision": precision, "rng_mode": rng_mode,
                 # chunk = a whole number of 148-SM waves of 128-point tiles (no partial last wave)
                 "max_points": (148 * 128 * 8 if wl.get("grid_dim") else 148 * 128 * 4 if wl["n_rays"] > 1000 else 32768)},
    }


class ClockSampler:
    """nvidia-smi sampled during the timed region (profiling recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def flops_per_point(E, Hd, B, units_only_chain=False):
    """SURVEY.md 8d: training step = 2*(6 F_MAC - 2 E Hd) with F_MAC = E Hd + 2B Hd^2 + (Hd+E) Hd + Hd."""
    f_mac = E * Hd + 2 * B * Hd * Hd + (Hd + E) * Hd + Hd
    return 2 * (6 * f_mac - 2 * E * Hd)


def host_threads():
    """One compute thread per PHYSICAL core this process may use (torch's own default; torchrun exports
    OMP_NUM_THREADS=1, which the CPU arm overrides).  Hyper-thread siblings are left idle: with 2 x 64 logical CPUs the
    reference step ran 2x slower and 3x noisier on 128 threads than on 64 (profiles/r02_summary.md)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        sib = open("/sys/devices/system/cpu/cpu0/topology/thread_siblings_list").read().strip()
        per_core = len(sib.replace("-", ",").split(",")) if sib else 1
        if "-" in sib:
            a, b = sib.split("-")[:2]
            per_core = int(b) - int(a) + 1
        n = max(1, n // max(per_core, 1))
    except Exception:
        pass
    torch.set_num_threads(n)
    return n


def make_cpu_stepper(wl, n_keyframes, n_rays=None):
    """The UNMODIFIED reference Trainer on device 'cpu' (oracle/_ref, or /root/reference in the build container),
    else the committed port.  -> (stepper, kind, description)"""
    from oracle import ref_shim
    cfg = make_config(wl, "fp32", "reference")
    if ref_shim.available():
        from oracle.ref_step import RefTrainerStepper
        st = RefTrainerStepper(cfg, n_keyframes=n_keyframes, n_rays=n_rays)
        return st, "reference", "unmodified isdf.modules.trainer.Trainer.step() on device 'cpu' (%s)" % st.trainer_file
    from oracle.cpu_step import CpuStepper

    class _Port:
        def __init__(self):
            self.s = CpuStepper(wl["H"], wl["W"], dict(fx=wl["fx"], fy=wl["fy"], cx=wl["cx"], cy=wl["cy"]),
                                n_frames=5, n_rays=n_rays or wl["n_rays"])

        def step(self):
            return self.s.step()
    return _Port(), "port", "oracle/cpu_step.py (torch CPU restatement of the reference step; reference package absent)"


def time_cpu(stepper, warmup, steps):
    for _ in range(warmup):
        stepper.step()
    per, pts = [], 0
    for _ in range(steps):
        t0 = time.perf_counter()
        _, n = stepper.step()
        per.append(time.perf_counter() - t0)
        pts += n
    return sum(per), pts, per


def run_reference_arm(args, wl, rank):
    """`--impl reference`: the reference's own CPU implementation of the step on this box's host cores (tier rule),
    same workload config, metric and unit as the B200 arm.  Rank 0 only; the other ranks exit without work."""
    if rank != 0:
        return
    cores = host_threads()
    S = wl["n_strat"] + wl["n_surf"]
    n_rays, sample = None, "full workload: every step is %d rays x %d samples" % (wl["n_rays"] * 5, S)
    if wl["n_rays"] * 5 * S > 2 * 27000:         # C4 / C5: a full step is minutes of CPU time -> bounded sample
        n_rays = max(8, 27000 // (5 * S))
        sample = "bounded sample: %d of %d rays/frame per step (%d points), same model / loss / window" % (
            n_rays, wl["n_rays"], n_rays * 5 * S)
    st, kind, what = make_cpu_stepper(wl, wl["keyframes"], n_rays)
    dt, pts, per = time_cpu(st, args.warmup, args.steps)
    val = pts / dt
    out = {"impl": "reference", "metric": "train ray-samples/sec", "value": val, "unit": "ray-samples/s",
           "iters_per_sec": args.steps / dt, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1000.0 * dt / args.steps, "ms_per_step_median": 1000.0 * statistics.median(per),
           "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": wl["name"], "device": "cpu", "points_per_step": pts // args.steps,
                      "keyframes": wl["keyframes"], "what": what},
           "cpu_baseline": {"value": val, "unit": "ray-samples/s", "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": val, "unit": "ray-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def load_traffic(precision, workload):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture of the same launch shape
    (profiles/chain_traffic.json, written by tools/update_traffic.py from an .ncu-rep; carries its provenance)."""
    f = os.path.join(ROOT, "profiles", "chain_traffic.json")
    try:
        rec = json.load(open(f)).get(precision, {}).get(workload)
    except Exception:
        return None, None
    if isinstance(rec, dict):
        return rec.get("dram_bytes_per_launch"), rec
    return rec, None


def run_grid_bench(args, wl, dev, rank, world, dist):
    """Row N1: Trainer.get_sdf_grid() -- K2 over the 200^3 lattice, points generated in the kernel.  One 'step' = one
    full grid evaluation; every rank evaluates the whole grid (replicas only: the grid is not sharded)."""
    import numpy as np
    from isdf.modules import trainer as trainer_mod
    np.random.seed(1)
    torch.manual_seed(1)
    cfg = make_config(wl, args.precision, "fast")
    tr = trainer_mod.Trainer(dev, cfg, incremental=True, grid_dim=wl["grid_dim"])
    T = np.eye(4)
    a = 0.3
    T[:2, :2] = [[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]]
    T[:3, 3] = [0.4, -0.2, 0.1]
    tr.set_scene_properties(T_extent_to_scene=T, bounds_extents=np.array([7.0, 3.2, 6.0]), scene_center=np.zeros(3))
    eng = tr.sdf_map.engine()
    n_pts = wl["grid_dim"] ** 3
    l0 = eng.launches
    tr.get_sdf_grid()
    launches_per_step = eng.launches - l0
    for _ in range(max(args.warmup, 3)):
        tr.get_sdf_grid()
    torch.cuda.synchronize(dev)
    if dist is not None:
        dist.barrier()
    sampler = ClockSampler(dev.index)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        grid = tr.get_sdf_grid()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    dump = {"sdf_grid": host_copy(grid)} if args.dump_outputs else None
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    # e2e: the public call + the grid on the host (32 MB D2H into pinned memory every step); no H2D (no inputs)
    host = torch.empty(wl["grid_dim"], wl["grid_dim"], wl["grid_dim"], dtype=torch.float32).pin_memory()
    e0.record()
    for _ in range(args.steps):
        host.copy_(tr.get_sdf_grid(), non_blocking=True)
        torch.cuda.synchronize(dev)
    e1.record()
    torch.cuda.synchronize(dev)
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    peaks = load_peaks()
    roof = None
    if eng.precision != "fp32":
        eng.profile(True)
        for _ in range(3):
            tr.get_sdf_grid()
        pr = eng.profile_read()
        eng.profile(False)
        n_l = max(pr["n_chain"], 1)
        pts_per_launch = 3.0 * n_pts / n_l
        fwd_flops_pt = 2.0 * 256 * 256 * (2 * wl["block"] + 3)          # 7 UMMA products per point (E padded to 256)
        chain_ms = pr["chain_ms"] / n_l
        ach = fwd_flops_pt * pts_per_launch / (chain_ms * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops", PEAKS_FALLBACK["bf16_tflops"])
        traffic, rec = load_traffic(eng.precision, "grid")
        roof = {"kernel": "tc_chain_kernel (forward-only program, 7 products per 128-point tile)", "bound": "tensor",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": traffic,
                "traffic_source": rec, "peak_source": peaks["_source"] + " burst bf16", "ms_per_launch": chain_ms,
                "points_per_launch": pts_per_launch, "algorithmic_flops_per_point": fwd_flops_pt,
                "algorithmic_bytes_per_point": 4}
    if rank == 0:
        out = {"metric": "sdf-grid points/sec (forward-only)", "value": world * n_pts * args.steps / (ms / 1e3),
               "unit": "points/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
               "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": eng.precision, "data": "synthetic (random-init weights)",
               "config": {"workload": wl["name"], "points_per_step_per_gpu": n_pts, "precision": eng.precision,
                          "parallelism": "replicas only (dp%d): every rank evaluates the whole lattice" % world,
                          "l2": "inputs are generated in-kernel; the 32 MB output per step is written once"},
               "clocks": clocks,
               "e2e": {"value": world * n_pts * args.steps / (e2e_ms / 1e3), "unit": "points/s",
                       "ms_per_step": e2e_ms / args.steps, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4 * n_pts,
                       "api": "Trainer.get_sdf_grid() + D2H of the [200,200,200] grid into pinned memory"},
               "gpu_launches": launches_per_step * args.steps, "roofline": roof, "cpu_baseline": None}
        print(json.dumps(out))
    if dump is not None:
        write_dump(args.dump_outputs, dump)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--precision", default=os.environ.get("ISDFB_PRECISION", "bf16x3g"),
                    choices=["bf16x3g", "bf16x3", "bf16", "fp32"])
    ap.add_argument("--workload", default="default", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the step's outputs (losses, sdf, loss matrix, parameters and "
                         "per-keyframe losses after the step; see reproducible_step) or, for the grid workload, the last "
                         "timed sdf grid as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or int(os.environ.get("WORLD_SIZE", 1)) > 1):
        ap.error("--dump-outputs records the B200 path of a single process")
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, wl, rank)
        return

    verbose = bool(os.environ.get("ISDFB_BENCH_VERBOSE"))

    def say(msg):
        if verbose:
            sys.stderr.write("[bench rank %d] %s\n" % (rank, msg))
            sys.stderr.flush()

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    say("process group ready")
    # the library __graft_entry__.build() compiled; the benchmark itself writes nothing into the tree
    from isdf_b200 import _lib
    _lib.load()
    say("library loaded")
    if args.workload == "grid":
        run_grid_bench(args, wl, dev, rank, world, dist)
        if dist is not None:
            dist.destroy_process_group()
        return
    tr = make_trainer(dev, wl, args.precision, rank, world, dist)
    say("keyframes resident")
    S = wl["n_strat"] + wl["n_surf"]
    rays_per_step = wl["n_rays"] * 5
    pts_per_step = rays_per_step * S
    eng = tr.sdf_map.engine()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # kernels of this library per step: counted on an eager (non-graph) step; the timed loop replays the
    # same launches from a CUDA graph, where the library's own counter cannot see them
    tr.use_graph = False
    tr.step(sync=False)
    l0 = eng.launches
    tr.step(sync=False)
    launches_per_step = eng.launches - l0
    tr.use_graph = True
    say("eager steps ok, %d launches/step" % launches_per_step)
    # ---------------- device-resident throughput (`value`) ----------------
    # warm-up: the W requested steps, plus what the graphed step needs before it is in steady state (the first step with
    # a new keyframe layout runs eagerly, the second is captured -- per gradient-buffer parity when data parallel -- and
    # the SM clocks need a few ms of load to settle): at least 30 steps in total, reported in config.warmup_internal
    n_warm = max(args.warmup, 3, 30)
    # nvidia-smi is started BEFORE the warm-up: its start-up (NVML initialisation, ~100 ms of driver calls) would otherwise
    # land inside a 20-step (12 ms) timed region; it then samples every 100 ms through warm-up and the timed region
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    for _ in range(n_warm):
        tr.step(sync=False)
    barrier()
    say("warm-up done")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        tr.step(sync=False)
    e1.record()
    torch.cuda.synchronize(dev)
    launches = launches_per_step * args.steps
    ms = e0.elapsed_time(e1)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * pts_per_step * args.steps / (ms_max / 1000.0)

    say("timed loop done: %.3f ms/step" % (ms_max / args.steps))
    # ---------------- end-to-end through the public API (`e2e`) ----------------
    # driver pattern of train.py:102-136: a new host frame is ingested every iters_per_frame steps
    # (pinned H2D of image+depth+pose, normals on device), every step's loss is read back (D2H).
    next_frame = rank + wl["keyframes"] * world
    h2d = 0
    # the host frames exist before the timed region (they stand in for decoded camera images); what is
    # timed per ingest is the pinned H2D copy, the normal estimation and the buffer update
    tr.scene_dataset.cache_frames = True
    N_E2E_WARM = 3
    for i in range(0, args.steps + N_E2E_WARM * tr.iters_per_frame, tr.iters_per_frame):
        _ = tr.scene_dataset[next_frame + (i // tr.iters_per_frame) * world]
    # warm-up of THIS path (untimed): three ingests with two synchronous steps each -- the first ingests after the
    # device-resident loop cost 15-40 ms of host time once (fresh device / page-locked allocations), which a 20-step
    # timed region would otherwise report as +1 ms per step
    for _w in range(N_E2E_WARM):     # three cycles: the device allocations of an ingest alternate between two generations
        fd = tr.get_data([next_frame])
        next_frame += world
        tr.last_is_keyframe = False
        tr.add_data(fd)
        for _ in range(2):
            losses, _ = tr.step()
            _ = float(losses["total_loss"])
    import gc
    gc.collect()              # BEFORE the barrier: a collection takes 10-20 ms and differs per rank
    barrier()
    step_ms, ingest_ms = [], []
    if not os.environ.get("ISDFB_BENCH_KEEP_GC"):
        gc.disable()          # a generation-2 collection (10-20 ms with torch + numpy loaded) inside a 13 ms timed region
                              # would be reported as +1 ms per step; collections resume right after the region
    e0.record()
    for i in range(args.steps):
        t0 = time.perf_counter()
        if i % tr.iters_per_frame == 0:
            fd = tr.get_data([next_frame])
            next_frame += world
            tr.last_is_keyframe = False            # replaces the live (non-key) frame, like add_frame
            tr.add_data(fd)
            h2d += fd.depth_batch_np.nbytes + fd.T_WC_batch_np.nbytes      # fast mode keeps the RGB image on the host
            t1 = time.perf_counter()
            ingest_ms.append(1e3 * (t1 - t0))
            t0 = t1
        losses, _ = tr.step()                      # the reference's call: synchronises and times the step (metrics.py)
        _ = float(losses["total_loss"])            # the step's loss, delivered D2H (pinned) by the step itself
        step_ms.append(1e3 * (time.perf_counter() - t0))
    e1.record()
    torch.cuda.synchronize(dev)
    gc.enable()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e_val = world * pts_per_step * args.steps / (e2e_ms / 1000.0)

    say("e2e loop done")
    # ---------------- roofline of the dominant kernel (rank 0, events inside the library) -------------
    roof = None
    peaks = load_peaks()
    prec = eng.precision                     # the model's actual precision (fp32 when the tcgen05 path refused the shape)
    if prec != "fp32":
        tr.use_graph = False                 # the event hooks live in the library's host code
        eng.profile(True)
        for _ in range(20):
            tr.step(sync=False)
        pr = eng.profile_read()                # 20 steps
        eng.profile(False)
        tr.use_graph = True
        lay_E = 3 + 2 * 21 * 6
        n_units = 4 * (2 * wl["block"] + 2) + 2                     # UMMA products of the chain kernel
        n_prof_steps = 20
        pts_per_launch = pts_per_step * n_prof_steps / max(pr["n_chain"], 1)    # a step is cut into max_points chunks
        tiles = int((pts_per_launch + 127) // 128)
        chain_flops = 2.0 * 256 * 256 * n_units * pts_per_launch     # algorithmic (real points, no padding / split passes)
        chain_ms = pr["chain_ms"] / max(pr["n_chain"], 1)
        dw_ms = pr["dw_ms"] / max(pr["n_dw"], 1)
        ach = chain_flops / (chain_ms * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops", PEAKS_FALLBACK["bf16_tflops"])
        roof = {"kernel": {"bf16x3": "tc_chain_kernel<3,1,false>", "bf16x3g": "tc_chain_kernel<3,1,true>",
                           "bf16": "tc_chain_kernel<1,1,false>"}[prec], "bound": "tensor",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "peak_source": peaks["_source"] + " burst bf16", "ms_per_launch": chain_ms,
                "algorithmic_flops_per_launch": chain_flops, "tiles": tiles,
                "dw_kernel_ms": dw_ms, "step_flops_per_point": flops_per_point(lay_E, wl["hidden"], wl["block"])}
        roof["traffic"], roof["traffic_source"] = load_traffic(prec, args.workload)
        if roof["traffic"]:
            # the same launch against the HBM roofline (ncu DRAM bytes / live kernel time): the kernel's second bound
            hbm_peak = peaks.get("hbm_gbs", PEAKS_FALLBACK["hbm_gbs"])
            roof["hbm_achieved_gbs"] = roof["traffic"] / (chain_ms * 1e-3) / 1e9
            roof["hbm_frac"] = roof["hbm_achieved_gbs"] / hbm_peak

    else:
        # fp32 CUDA-core path (models the tcgen05 kernels do not take, e.g. hidden 512): whole-step figure against the
        # same tensor peak the north-star names -- the register-tiled SGEMM cannot approach it; reported, not hidden
        lay_E = 3 + 2 * 21 * 6
        fpp = flops_per_point(lay_E, wl["hidden"], wl["block"])
        ach = fpp * pts_per_step / (ms_max / args.steps * 1e-3) / 1e12
        peak = peaks.get("bf16_tflops", PEAKS_FALLBACK["bf16_tflops"])
        roof = {"kernel": "sgemm_kernel + element-wise kernels (fp32 CUDA-core path, simt_path.cu), whole step",
                "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": None,
                "peak_source": peaks["_source"] + " burst bf16", "step_flops_per_point": fpp,
                "note": "fp32 FFMA peak of the part is ~74 TFLOP/s (148 SMs x 128 lanes x 2 x 1.965 GHz): %.0f %% of that"
                        % (100.0 * ach / 74.4)}

    # ---------------- data-parallel parity (N > 1): replicas identical, fused exchange == NCCL all-reduce -----------
    xchg = None
    used_multicast = tr._xchg is not None
    if world > 1:
        flat = tr.sdf_map.flat_parameters()
        ref0 = flat.clone()
        dist.broadcast(ref0, 0)
        dmax = (flat - ref0).abs().max().reshape(1).double()
        dist.all_reduce(dmax, op=dist.ReduceOp.MAX)
        xchg = {"replica_param_max_abs_diff_vs_rank0": float(dmax.item()), "param_max_abs": float(flat.abs().max().item()),
                "steps_taken": int(tr.optimiser.step_count)}
        if tr._xchg is not None and tr._last_pts is not None:
            # the same per-rank batch (this rank's last sampled rays) through both exchanges: the multimem.red flush
            # of the weight-gradient kernel, then -- exchange uninstalled -- a plain NCCL all-reduce of the local sums
            pts, lc = tr._last_pts
            scratch = torch.zeros(4, dtype=torch.float32, device=dev)

            def k4():
                eng.train_fwd_bwd(pts["pc"], pts["z_vals"], pts["depth_sample"], pts["dirs_C_sample"], pts["T_WC_sample"],
                                  pts["norm_sample"], pts["noise"], lc, ray_valid=pts["ray_valid"], want_grad=False,
                                  loss_sums=scratch)
            par = tr._xchg.parity
            eng.select_grad_buffer(par)
            k4()
            eng.zero_grad_buffer(1 - par)
            tr._xchg.barrier()
            fused = eng.grad_buffer().clone()
            barrier()
            tr._xchg.close()
            eng.zero_grad()
            k4()
            summed = eng.grad_buffer().clone()
            dist.all_reduce(summed)
            err = ((fused - summed).abs().max() / summed.abs().max()).reshape(1).double()
            dist.all_reduce(err, op=dist.ReduceOp.MAX)
            xchg["fused_vs_nccl_grad_max_rel_diff"] = float(err.item())
            tr._xchg = None
        barrier()

    # ---------------- CPU baseline: the reference's own step on this box's host cores (bounded sample) ----------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        cores = host_threads()
        n_r = min(wl["n_rays"], 200)
        st, kind, what = make_cpu_stepper(wl, 5, n_r)
        dt, pts, per = time_cpu(st, 1, 5)
        cpu = {"value": pts / dt, "unit": "ray-samples/s", "cores": cores, "kind": kind,
               "sample": "5 steps of %d rays x %d samples after 1 warm-up; %s" % (n_r * 5, S, what),
               "iters_per_sec": 5 / dt, "ms_per_step_median": 1000.0 * statistics.median(per)}

    if args.dump_outputs:           # before the result line, which stays the last line on stdout
        write_dump(args.dump_outputs, reproducible_step(dev, wl, args.precision))
    if rank == 0:
        out = {"metric": "train ray-samples/sec", "value": value, "unit": "ray-samples/s",
               "iters_per_sec": world * args.steps / (ms_max / 1000.0) / world,
               "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
               "dtype": {"bf16x3": "bf16x3 (bf16 hi/lo split, fp32 accumulate)",
                         "bf16x3g": "bf16x3 (bf16 hi/lo split, fp32 accumulate; weight-gradient operands single bf16)",
                         "bf16": "bf16", "fp32": "f32"}[prec],
               "data": "synthetic",
               "config": {"workload": wl["name"], "warmup_internal": n_warm, "rays_per_step_per_gpu": rays_per_step,
                          "samples_per_ray": S,
                          "points_per_step_per_gpu": pts_per_step, "keyframes_per_gpu": wl["keyframes"],
                          "precision": prec, "rng_mode": "fast (fixed shapes, validity mask, no host sync; whole step replayed as one CUDA graph)",
                          "parallelism": "dp%d (keyframe-sharded; gradient exchange: %s)" % (world, (
                              "none" if world == 1 else
                              "fused into the weight-gradient kernel over NVLink multicast (multimem.red) + 1 barrier" if used_multicast
                              else "one NCCL all-reduce of the packed gradient%s" % (" inside the step graph" if tr._nccl_in_graph else ""))),
                          "l2": "no explicit flush: keyframe buffer %.0f MB and per-step side state %.0f MB both exceed the 126 MB L2"
                                % (wl["keyframes"] * wl["H"] * wl["W"] * 16 / 1e6, pts_per_step * 0.041)},
               "clocks": clocks,
               "e2e": {"value": e2e_val, "unit": "ray-samples/s", "ms_per_step": e2e_ms / args.steps,
                       "step_ms_median": statistics.median(step_ms),
                       "ingest_ms_median": statistics.median(ingest_ms) if ingest_ms else None,
                       "ingest_ms_max": max(ingest_ms) if ingest_ms else None, "step_ms_max": max(step_ms),
                       "ingest_every_steps": tr.iters_per_frame,
                       "h2d_bytes_per_step": h2d / args.steps, "d2h_bytes_per_step": 16,
                       "api": "isdf.modules.trainer.Trainer.get_data/add_data/step() + float(losses['total_loss'])"},
               "gpu_launches": launches,
               "roofline": roof, "cpu_baseline": cpu, "exchange_parity": xchg}
        print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
