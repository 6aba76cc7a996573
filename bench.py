#!/usr/bin/env python
"""bench.py — LM iterations/s of the LiDAR-visual BA hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config C] [--dump-outputs DIR]

A *step* — the same for both arms, written into `config.step` of both lines — is ONE full LM iteration of the whole hot path on
one synthetic problem, started from the initial state (SURVEY.md §8d):
    t_A  one BALM2 pass  = Hessian/gradient build + damped block-LDL^T solve + retraction
                           + residual-only pass + accept/reject          (bavoxel.hpp:686-766)
    t_B  one Ceres-style pass = Jacobians + Schur elimination + reduced solve + back-substitution
                           + candidate cost + accept/reject              (src/lvba_system.cpp:1643)
    metric value = 1 / (t_A + t_B)            [LM iterations / s]
`value`: inputs resident in HBM (device-to-device restore of the initial state before every step).
`e2e`:   the call a user of the reference makes: ONE call of each boundary with HOST (pinned) buffers to the reference's own caps
         (BALM2::damping_iter <= 10 passes, ceres::Solve <= 50 passes, default stop tests) through lvba_lidar_lm / lvba_visual_lm;
         validation, symbolic set-up, H2D upload of the whole problem, all passes and the D2H result copy are inside the timed
         region of every call; t_A, t_B = call time / passes executed.  The CPU arm's `e2e` is the same call of its own code.
`one_pass_call` (informational): the same ABI calls limited to one pass (set-up and upload not amortised).

Workload: N = 1 -> BASELINE.json configs[2] (2000 poses / 200k plane voxels / 100k tracks, the config the metric is quoted on);
N > 1 -> configs[4] (5000 / 500k / 300k, the config BASELINE names for scaling), sharded by contiguous pose-block rows; the
N > 1 line also carries `n1_same_config`: the same config measured on ONE GPU by rank 0 in the same run, so that a like-for-like
efficiency can be formed.  `--config` overrides.

`--impl reference` times the reference-restated CPU path (oracle/cpu_ref.cpp — the reference itself needs Eigen/Ceres/PCL/ROS and
cannot be built here) on the box's host cores, same step / config / metric.  Path A runs with the thread count that is fastest
in a sweep that always includes the reference's own fixed 16 (bavoxel.hpp:25); path B likewise (Ceres uses all threads).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "LM iterations/sec (Jacobian+Hessian build + Schur solve)"
UNIT = "LM iterations/s"
VKEYS = ("q", "t", "X", "plane_nd", "obs_ptr", "obs_cam", "obs_uv", "intr", "sigma_px", "sigma_plane")
STEP_TEXT = ("value: one full LM iteration from the initial state — path A (Hessian build + damped LDL^T solve + retraction + residual "
             "pass + accept test) then path B (Jacobians + Schur + reduced solve + back-substitution + candidate cost); "
             "e2e: one call of each boundary as the reference makes it, from host buffers (damping_iter to <= 10 passes, the Ceres solve to "
             "<= 50 passes, default stop tests), wall time / passes executed, t_A + t_B")
L2_TEXT = "GPU arm: 256 MiB buffer written between timed steps (L2 flush); CPU arm: per-step working set (>300 MB) exceeds the host LLC"
FP64_PEAK_TFLOPS = 148 * 63.7 * 2 * 1.965e9 / 1e12      # measured 63.7 DFMA/clk/SM (tools/ubench/fp64_rate.cu) x 148 SMs x 1.965 GHz


def workload_name(cfg, p):
    return (f"config {cfg}: {p['n_poses']} poses / {p['n_vox']} plane voxels / {p['n_tracks']} visual tracks, "
            f"synthetic (oracle/synth.py, seed {p['seed']})")


def config_block(cfg, p):
    """identical in both arms (the driver compares it)"""
    return {"workload": workload_name(cfg, p), "step": STEP_TEXT, "l2": L2_TEXT}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 9 for i in range(4) if r[5 + i].lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def algorithmic_bytes(p, lid_counts, vis_counts, n_active):
    """SURVEY.md §8(d) formulas evaluated exactly on the generated instance."""
    W = p["n_poses"]
    nnzA, nbH = lid_counts["nnz"], lid_counts["n_blocks_nonzero"]
    build_A = 84 * nnzA + 96 * W + 288 * nbH + 48 * W            # Hessian pass: read slots + poses, write H, g
    resid_A = 84 * nnzA + 96 * W
    nnzB, Tv, nbS = vis_counts["nnz_valid"], vis_counts["n_valid_tracks"], vis_counts["n_blocks_env"]
    bytes_B = 2 * (16 * nnzB + 56 * p["n_poses"] + 56 * Tv) + 288 * nbS + 48 * n_active + 24 * Tv
    return dict(lidar_build=build_A, lidar_residual=resid_A, bytes_A=build_A + resid_A, bytes_B=bytes_B)


# ------------------------------------------------------------------------------------------------ CPU arm
def step_outputs(poses, a, q, t, X, b):
    """what one step hands its caller, under the names --dump-outputs writes; a, b: the two paths' summaries"""
    return {"lidar_poses": poses, "lidar_cost": np.array([a["cost_first"], a["cost_last"]]),
            "visual_q": q, "visual_t": t, "visual_X": X, "visual_cost": np.array([b["cost_first"], b["cost_last"]])}


def dump_outputs(out_dir, outputs):
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, a in outputs.items():
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a, np.float64))


def cpu_pass(p, threads_a, threads_b):
    """one full LM pass of each path on the full problem with the CPU restatement; ms per pass (A, B) and step_outputs"""
    from oracle import cpu_ref
    poses, a = cpu_ref.lidar_lm(p["vox_ptr"], p["pose_idx"], p["clusters"], p["poses"], max_iter=1, rel_tol=-1.0, threads=threads_a)
    q, t, X, b = cpu_ref.visual_lm(*[p[k] for k in VKEYS], max_iter=1, threads=threads_b, function_tolerance=-1.0)
    tA = a["ms_build"] + a["ms_solve"] + a["ms_residual"]
    tB = b["ms_build"] + b["ms_solve"] + b["ms_residual"]
    return tA, tB, step_outputs(poses, a, q, t, X, b)


def cpu_thread_sweep(p):
    """fastest thread count per path; the reference's fixed 16 (bavoxel.hpp:25) is always a candidate"""
    from oracle import cpu_ref
    hw = cpu_ref.hardware_threads()
    cand = sorted({t for t in (8, 16, 32, 64, hw) if t <= max(hw, 16)})
    sweep = {}
    for t in cand:
        tA, tB, _ = cpu_pass(p, t, t)
        sweep[str(t)] = {"ms_A": round(tA, 1), "ms_B": round(tB, 1)}
    best_a = min(cand, key=lambda t: sweep[str(t)]["ms_A"])
    best_b = min(cand, key=lambda t: sweep[str(t)]["ms_B"])
    return best_a, best_b, sweep, hw


def run_reference(args, p, cfg):
    """--impl reference: the CPU path on the host cores, same step / metric / config."""
    ta, tb, sweep, hw = cpu_thread_sweep(p)
    times = []
    for i in range(args.warmup + args.steps):
        tA, tB, outputs = cpu_pass(p, ta, tb)
        if i >= args.warmup:
            times.append((tA + tB) / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    mean = sum(times) / len(times)
    val = 1.0 / mean
    # e2e of this arm: the same call of each boundary to the reference's caps, time / passes (host memory only: no copies)
    from oracle import cpu_ref
    n_calls = 2
    e2e_s, info = 0.0, {}
    for _ in range(n_calls):
        t0 = time.perf_counter()
        _, a = cpu_ref.lidar_lm(p["vox_ptr"], p["pose_idx"], p["clusters"], p["poses"], threads=ta)
        t1 = time.perf_counter()
        _, _, _, b = cpu_ref.visual_lm(*[p[k] for k in VKEYS], threads=tb)
        t2 = time.perf_counter()
        e2e_s += (t1 - t0) / max(a["iterations"], 1) + (t2 - t1) / max(b["iterations"], 1)
        info = {"ms_call_A": (t1 - t0) * 1e3, "ms_call_B": (t2 - t1) * 1e3, "passes_A": int(a["iterations"]), "passes_B": int(b["iterations"]),
                "hessian_builds_A": int(a["builds"]), "cost_A": a["cost_last"], "cost_B": b["cost_last"]}
    e2e_val = n_calls / e2e_s
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": mean * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(cfg, p),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": max(ta, tb), "threads_path_A": ta, "threads_path_B": tb,
                             "host_hardware_threads": hw, "kind": "port", "thread_sweep_ms_per_pass": sweep,
                             "sample": "each step = 1 full LM pass of path A + 1 of path B on the full problem (oracle/cpu_ref.cpp: the reference "
                                       "restated; Eigen/Ceres are not installable here)",
                             "why_port": "the reference's own source does compile (oracle/_ref, on stand-in library headers) and the port is held against it — H 4.6e-11, g 1.3e-11 at this config, the whole damping_iter at config B (profiles/r02_ref_pin_scale_*.txt) — but BALM2::damping_iter as written keeps vector<PointCluster>(win_size) per voxel and 19 dense 6W x 6W matrices: 42 GB + 22 GB and minutes per pass at 2000 poses, on our eager stand-in for Eigen; the port (CSR slots, block envelope, the reference's thread model) is the faster, fairer opponent"},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "calls_timed": n_calls, **info,
                    "step": "one full call of each boundary to the reference's caps (<= 10 / <= 50 passes), time / passes executed"},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def measure_resident(pkg, torch, p, device, steps, warmup, barrier, rank):
    """K timed steps with inputs resident; returns dict with host seconds, per-phase device ms, launches, full-LM summaries"""
    L = pkg.LidarProblem(p["vox_ptr"], p["pose_idx"], p["clusters"], p["poses"], device=device)
    Vz = pkg.VisualProblem(*[p[k] for k in VKEYS], device=device)
    lo_opts = pkg.lidar_default_opts(); lo_opts.rel_tol = -1.0; lo_opts.max_iter = 1 << 30
    vo_opts = pkg.visual_default_opts(); vo_opts.function_tolerance = -1.0; vo_opts.parameter_tolerance = -1.0
    vo_opts.gradient_tolerance = -1.0; vo_opts.max_iter = 1 << 30
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")      # > 126 MB L2

    def one_step():
        flush.fill_(rank + 1)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        L.reset_lm(lo_opts); L.reset_state(); sa = L.iterate(1)
        Vz.reset_lm(vo_opts); Vz.reset_state(); sb = Vz.iterate(1)
        return time.perf_counter() - t0, sa, sb

    for _ in range(warmup):
        one_step()
    barrier()
    pkg.comm_bytes_sent()                                            # reset the NCCL payload counter
    wall0 = time.perf_counter()
    host_s, launches = 0.0, 0
    dev_ms = {"build_A": 0.0, "solve_A": 0.0, "resid_A": 0.0, "build_B": 0.0, "solve_B": 0.0, "resid_B": 0.0}
    for _ in range(steps):
        dt, sa, sb = one_step()
        host_s += dt
        dev_ms["build_A"] += sa["ms_build"]; dev_ms["solve_A"] += sa["ms_solve"]; dev_ms["resid_A"] += sa["ms_residual"]
        dev_ms["build_B"] += sb["ms_build"]; dev_ms["solve_B"] += sb["ms_solve"]; dev_ms["resid_B"] += sb["ms_residual"]
        launches += sa["kernel_launches"] + sb["kernel_launches"]
    barrier()
    wall = time.perf_counter() - wall0
    nccl_bytes = pkg.comm_bytes_sent() / steps
    q, t, X = Vz.get_state()                                     # what the last timed step left, before the full LM below moves it
    outputs = step_outputs(L.get_poses(), sa, q, t, X, sb)
    ra, rb = L.owned_rows(), Vz.owned_rows()
    # full LM to the reference's caps (BASELINE configs[2]), device resident
    L.reset_lm(None); L.reset_state(); fa2 = L.iterate(2)        # the LM amplifies rounding differences from iteration to iteration
    L.reset_lm(None); L.reset_state(); fa = L.iterate(10)        # (profiles/r02_lm_sensitivity_*.txt): parity across GPU counts is
    Vz.reset_lm(None); Vz.reset_state(); fb = Vz.iterate(50)     # checked after 2 iterations, the full-call costs are reported
    out = {"cost_A_after_2": fa2["cost_last"],"host_s": host_s, "wall": wall, "launches": launches, "dev_ms": {k: v / steps for k, v in dev_ms.items()},
           "full_A": fa, "full_B": fb, "lid_counts": L.counts(nonzero=True), "vis_counts": Vz.counts(),
           "n_active": len(Vz.structure()[0]), "structA": L.structure(), "structB": Vz.structure(),
           "nccl_bytes_per_step": nccl_bytes, "owned_rows_A": ra, "owned_rows_B": rb, "outputs": outputs}
    L.close(); Vz.close()
    del flush
    return out


def ldl_flops(brow, bcol, n):
    below = np.bincount(bcol[brow > bcol], minlength=n).astype(np.float64)     # blocks under every pivot
    return float((below * (below + 1) / 2 * 432 + below * 72 * 2 + below * 72 * 2).sum())   # trailing update + scale + two substitutions


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=["A", "B", "C", "E"])
    ap.add_argument("--e2e-steps", type=int, default=3, help="timed full ABI calls of each boundary (after one warm-up call)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the GPU-vs-CPU full-LM parity check at the benchmarked config")
    ap.add_argument("--no-voxel-map", action="store_true", help="skip the boundary-B3 (voxel map) side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed (poses, cameras, points, costs) as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = args.config or ("C" if world == 1 else "E")

    from oracle import synth
    if args.impl == "reference":
        if rank != 0:
            return 0
        p = synth.make_config(cfg)
        run_reference(args, p, cfg)
        return 0

    import torch
    import torch.distributed as dist
    import __graft_entry__ as graft
    pkg = graft.load_package()
    pkg.load_library()
    if pkg.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device — the LVBA hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    p = synth.make_config(cfg)                            # identical on every rank (counter-based RNG)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    n1 = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # the same config on ONE GPU, measured by rank 0 before the communicator exists (the others wait)
        if rank == 0:
            r1 = measure_resident(pkg, torch, p, local_rank, max(5, args.steps // 2), 3, lambda: torch.cuda.synchronize(), 0)
            n1 = {"value": max(5, args.steps // 2) / r1["host_s"], "device_ms_per_step": r1["dev_ms"], "cost_A_after_2": r1["cost_A_after_2"],
                  "full_lm_cost_A": r1["full_A"]["cost_last"], "full_lm_cost_B": r1["full_B"]["cost_last"]}
        dist.barrier()
        uid = [pkg.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        pkg.comm_init(world, rank, uid[0], local_rank)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    R = measure_resident(pkg, torch, p, local_rank, args.steps, args.warmup, barrier, rank)
    clocks = sampler.stop() if rank == 0 else None
    dev_total_ms = sum(R["dev_ms"].values())
    tt = torch.tensor([R["host_s"], dev_total_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    host_s_max, dev_ms_max = tt[0].item(), tt[1].item()
    ms_per_step = host_s_max * 1e3 / args.steps
    value = args.steps / host_s_max

    # ---- e2e: the same step through the one-shot C-ABI calls, host (pinned) buffers, everything inside the timed region
    def pinned(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        return t.numpy()
    hp = {k: pinned(p[k]) for k in ("vox_ptr", "pose_idx", "clusters", "poses", "q", "t", "X", "plane_nd", "obs_ptr", "obs_cam", "obs_uv", "intr")}
    o1 = pkg.lidar_default_opts(); o1.max_iter = 1; o1.rel_tol = -1.0; o1.device = local_rank
    v1 = pkg.visual_default_opts(); v1.max_iter = 1; v1.function_tolerance = -1.0; v1.parameter_tolerance = -1.0; v1.gradient_tolerance = -1.0
    v1.device = local_rank
    oF = pkg.lidar_default_opts(); oF.device = local_rank
    vF = pkg.visual_default_opts(); vF.device = local_rank

    def abi_calls(lo, vo):
        barrier()
        t0 = time.perf_counter()
        _, sa = pkg.lidar_lm(hp["vox_ptr"], hp["pose_idx"], hp["clusters"], hp["poses"], lo)
        t1 = time.perf_counter()
        _, _, _, sb = pkg.visual_lm(hp["q"], hp["t"], hp["X"], hp["plane_nd"], hp["obs_ptr"], hp["obs_cam"], hp["obs_uv"], hp["intr"],
                                    p["sigma_px"], p["sigma_plane"], opts=vo)
        t2 = time.perf_counter()
        return t1 - t0, t2 - t1, sa, sb

    n_e2e = max(1, args.e2e_steps)
    e2e_s, h2d, d2h, call_s = 0.0, 0.0, 0.0, [0.0, 0.0]
    for i in range(n_e2e + 1):                                   # first call is warm-up
        ta, tb, sa, sb = abi_calls(oF, vF)
        if i > 0:
            pa, pb = max(sa["iterations"], 1), max(sb["iterations"], 1)
            e2e_s += ta / pa + tb / pb
            h2d += sa["h2d_bytes"] / pa + sb["h2d_bytes"] / pb; d2h += sa["d2h_bytes"] / pa + sb["d2h_bytes"] / pb
            call_s[0] += ta; call_s[1] += tb
    te = torch.tensor([e2e_s / n_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = 1.0 / te.item()
    full_call = {"ms_call_A": call_s[0] * 1e3 / n_e2e, "ms_call_B": call_s[1] * 1e3 / n_e2e, "passes_A": sa["iterations"], "passes_B": sb["iterations"],
                 "hessian_builds_A": sa["hessian_builds"], "h2d_bytes_per_call": sa["h2d_bytes"] + sb["h2d_bytes"],
                 "d2h_bytes_per_call": sa["d2h_bytes"] + sb["d2h_bytes"], "cost_A": sa["cost_last"], "cost_B": sb["cost_last"]}
    ta, tb, sa1, sb1 = abi_calls(o1, v1)                         # warm-up of the one-pass variant
    ta, tb, sa1, sb1 = abi_calls(o1, v1)
    one_pass_call = {"value": 1.0 / (ta + tb), "ms_call_A": ta * 1e3, "ms_call_B": tb * 1e3,
                     "note": "lvba_lidar_lm(max_iter=1) + lvba_visual_lm(max_iter=1): set-up and upload of the whole problem for ONE pass"}

    rc = 0
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, R["outputs"])
    if rank == 0:
        ab = algorithmic_bytes(p, R["lid_counts"], R["vis_counts"], R["n_active"])
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()); peak = float(peaks["hbm_gbs"]); peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        prof = {}
        try:     # DRAM bytes per launch from the committed `ncu --set full` captures (config C, one GPU)
            prof = json.loads((ROOT / "profiles" / "r02_ncu_summary.json").read_text())
        except Exception:
            try:
                prof = json.loads((ROOT / "profiles" / "r01_ncu_full_summary.json").read_text())
            except Exception:
                prof = {}

        def traffic_of(kernel):
            try:
                if cfg == "C" and world == 1:
                    return (float(prof[kernel]["dram__bytes_read.sum"]) + float(prof[kernel]["dram__bytes_write.sum"])) * 1e6
            except Exception:
                pass
            return None
        dm = R["dev_ms"]
        # the largest single kernel of the step is the Hessian build of path A (one launch); the solves are ~30 launches each
        build_ms = dm["build_A"]
        achieved = ab["lidar_build"] / (build_ms * 1e-3) / 1e9
        roofline = {"kernel": "lidar_build_kernel (largest single kernel of the step; timed with the memset of H and the partial-sum reduce)",
                    "share_of_step": build_ms / max(dev_total_ms, 1e-9),
                    "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic_of("lidar_build_kernel"), "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": ab["lidar_build"], "avg_launch_ms": build_ms,
                    "fp64_tflops": 3.6e9 * (p["n_vox"] / 200000.0) / (build_ms * 1e-3) / 1e12, "fp64_frac_of_chip": 3.6e9 * (p["n_vox"] / 200000.0) / (build_ms * 1e-3) / 1e12 / FP64_PEAK_TFLOPS,
                    "note": "CUDA events on the library's launch stream; ncu: atomic (RED.ADD.F64) / shared-memory bound, not HBM bound (DESIGN.md 4)"}
        resid_ms = dm["resid_A"]
        roofline_residual = {"kernel": "lidar_residual_kernel (+ retraction, partial-sum reduce)", "bound": "hbm",
                             "achieved": ab["lidar_residual"] / (resid_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": ab["lidar_residual"] / (resid_ms * 1e-3) / 1e9 / peak, "traffic": traffic_of("lidar_residual_kernel"),
                             "avg_launch_ms": resid_ms}
        brA, bcA = R["structA"]
        sv = R["structB"]
        flA = ldl_flops(np.asarray(brA), np.asarray(bcA), p["n_poses"])
        flB = ldl_flops(np.asarray(sv[1]), np.asarray(sv[2]), R["n_active"])
        solve_s = (dm["solve_A"] + dm["solve_B"]) * 1e-3
        roofline_solve = {"kernels": "substructured block LDL^T: env_factor_la_kernel (chunk interiors, grid = chunks), nd_dense_factor_kernel "
                                     "(separators), nd_spike_kernel, nd_syrk_kernel, env_backsolve_warp_kernel (csrc/nd_solver.cuh)",
                          "share_of_step": (dm["solve_A"] + dm["solve_B"]) / max(dev_total_ms, 1e-9),
                          "bound": "fp64 (latency of the pivot chains; no HBM traffic to speak of: the systems are L2 resident)",
                          "fp64_flops_sequential_ldlt": flA + flB, "achieved_tflops": (flA + flB) / solve_s / 1e12,
                          "peak_tflops_chip": FP64_PEAK_TFLOPS, "frac": (flA + flB) / solve_s / 1e12 / FP64_PEAK_TFLOPS,
                          "note": "useful flops = those of ONE sequential banded LDL^T (the substructured solve spends ~4x more on spikes "
                                  "and separator updates); denominator = whole-chip FP64 vector peak"}
        step_bytes = ab["bytes_A"] + ab["bytes_B"]
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config_block(cfg, p),
                "run": {"parallelism": f"pose-block-row shards x{world}", "config_letter": cfg,
                        "row_owned_system": bool(R["owned_rows_A"][2]), "rank0_rows_A": list(R["owned_rows_A"][:2]), "rank0_rows_B": list(R["owned_rows_B"][:2]),
                        "nccl_payload_bytes_per_step_rank0": R["nccl_bytes_per_step"],
                        "scale_config": "N = 1: config C (headline); N > 1: config E, with n1_same_config measured in the same run"},
                "device_ms_per_step": dm,
                "device_ms_per_step_total_max_over_ranks": dev_ms_max / args.steps,
                "timed_region_wall_s": R["wall"],
                "roofline": roofline, "roofline_residual": roofline_residual, "roofline_solve": roofline_solve,
                "step_hbm": {"algorithmic_bytes": step_bytes, "achieved_gbs": step_bytes / (ms_per_step * 1e-3) / 1e9,
                             "frac_of_peak": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak},
                "algorithmic_bytes": ab,
                "full_lm": {"A": {k: R["full_A"][k] for k in ("iterations", "accepted", "cost_first", "cost_last", "ms_total")},
                            "B": {k: R["full_B"][k] for k in ("iterations", "accepted", "cost_first", "cost_last", "ms_total")}},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d / n_e2e), "d2h_bytes_per_step": int(d2h / n_e2e),
                        "step": "one lvba_lidar_lm call (<= 10 passes) + one lvba_visual_lm call (<= 50 passes) from pinned host buffers: "
                                "validation, symbolic set-up, H2D of the whole problem, the passes, D2H inside the timed region; "
                                "t = call time / passes executed; bytes per step = bytes per call / passes",
                        "calls_timed": n_e2e, **full_call},
                "one_pass_call": one_pass_call,
                "gpu_launches": int(R["launches"]), "clocks": clocks}
        if n1 is not None:
            line["n1_same_config"] = n1
            line["efficiency_vs_n1_same_config"] = value / (world * n1["value"])
            pv = {"rel_A_after_2_iterations": abs(R["cost_A_after_2"] - n1["cost_A_after_2"]) / abs(n1["cost_A_after_2"]),
                  "rel_B_full_call": abs(R["full_B"]["cost_last"] - n1["full_lm_cost_B"]) / abs(n1["full_lm_cost_B"]),
                  "rel_A_full_call_informational": abs(R["full_A"]["cost_last"] - n1["full_lm_cost_A"]) / abs(n1["full_lm_cost_A"]),
                  "note": "path A of this config is chaotic beyond ~6 LM iterations even between two runs on ONE GPU (RED.ADD order; "
                          "profiles/r02_lm_sensitivity_E.txt), so the gate is the cost after 2 iterations + the full call of path B"}
            pv["ok"] = bool(pv["rel_A_after_2_iterations"] <= 1e-6 and pv["rel_B_full_call"] <= 1e-6)
            line["parity_vs_n1"] = pv
            if not pv["ok"]:
                rc = 3
        if world == 1 and not args.no_cpu_baseline:
            ta_, tb_, sweep, hw = cpu_thread_sweep(p)
            tA, tB, _ = cpu_pass(p, ta_, tb_)
            line["cpu_baseline"] = {"value": 1e3 / (tA + tB), "unit": UNIT, "cores": max(ta_, tb_), "threads_path_A": ta_, "threads_path_B": tb_,
                                    "host_hardware_threads": hw, "kind": "port", "thread_sweep_ms_per_pass": sweep,
                                    "sample": "1 full LM pass of path A + 1 of path B on the full problem (oracle/cpu_ref.cpp) at the fastest thread "
                                              "count of the sweep (the reference's fixed 16 included)", "ms_A": tA, "ms_B": tB,
                                    "why_port": "the reference's own source does compile (oracle/_ref, on stand-in library headers) and the port is held against it — H 4.6e-11, g 1.3e-11 at this config, the whole damping_iter at config B (profiles/r02_ref_pin_scale_*.txt) — but BALM2::damping_iter as written keeps vector<PointCluster>(win_size) per voxel and 19 dense 6W x 6W matrices: 42 GB + 22 GB and minutes per pass at 2000 poses, on our eager stand-in for Eigen; the port (CSR slots, block envelope, the reference's thread model) is the faster, fairer opponent"}
            if not args.no_parity:
                # north-star check at the benchmarked config: full LM (caps 10 / 50) on the GPU against the CPU restatement
                from oracle import cpu_ref
                t0 = time.perf_counter()
                _, ca = cpu_ref.lidar_lm(p["vox_ptr"], p["pose_idx"], p["clusters"], p["poses"], threads=ta_)
                _, _, _, cb = cpu_ref.visual_lm(*[p[k] for k in VKEYS], threads=tb_)
                relA = abs(R["full_A"]["cost_last"] - ca["cost_last"]) / abs(ca["cost_last"])
                relB = abs(R["full_B"]["cost_last"] - cb["cost_last"]) / abs(cb["cost_last"])
                ok = bool(relA <= 1e-6 and relB <= 1e-6)
                line[f"parity_{cfg}"] = {"tolerance_rel": 1e-6, "ok": ok,
                                         "A": {"gpu_cost": R["full_A"]["cost_last"], "cpu_cost": ca["cost_last"], "rel": relA,
                                               "gpu_iterations": R["full_A"]["iterations"], "cpu_iterations": int(ca["iterations"])},
                                         "B": {"gpu_cost": R["full_B"]["cost_last"], "cpu_cost": cb["cost_last"], "rel": relB,
                                               "gpu_iterations": R["full_B"]["iterations"], "cpu_iterations": int(cb["iterations"])},
                                         "cpu_full_call": {"ms_per_pass_A": ca["ms_total"] / max(ca["iterations"], 1), "ms_per_pass_B": cb["ms_total"] / max(cb["iterations"], 1),
                                                           "value": 1e3 / (ca["ms_total"] / max(ca["iterations"], 1) + cb["ms_total"] / max(cb["iterations"], 1))},
                                         "seconds": time.perf_counter() - t0}
                if not ok:
                    rc = 3
        if world == 1 and not args.no_voxel_map:
            # Boundary B3 (set-up stage, DESIGN.md 4.3) measured OUTSIDE the timed region, in a child process so that
            # nothing it does can disturb the numbers above; reported next to them, not part of `value` / `e2e`.
            try:
                r = subprocess.run([sys.executable, str(ROOT / "tools" / "bench_voxel_map.py")], capture_output=True, text=True, timeout=300)
                last = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
                line["voxel_map"] = json.loads(last[-1]) if last else {"error": (r.stderr or r.stdout)[-400:], "rc": r.returncode}
            except Exception as e:          # noqa: BLE001 - a side measurement must never take the bench line down
                line["voxel_map"] = {"error": repr(e)[:400]}
        print(json.dumps(line), flush=True)
    if world > 1:
        pkg.comm_destroy()
        dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
