#!/usr/bin/env python
"""bench.py -- BA iterations/sec of the BALM 2.0 hot path on B200 (BASELINE.json metric).

A "step" is one Levenberg-Marquardt iteration of BALM2::damping_iter (bavoxel.hpp:1104-1157):
  1 Hessian/gradient evaluation (left_evaluate_acc2) + 1 damped LDL^T solve + SE(3) left update
  + 1 residual-only evaluation, with the Hessian re-evaluated every iteration (force_hess) so that every step
  is the same amount of work whether the trial step is accepted or not.
Workload (N=1): BASELINE config C3 -- 500 poses x 100 000 plane voxels, synthetic plane features of the
benchmark_virtual shape (benchmark_virtual.cpp:547-606), every pose sees every plane, 40 points/observation.
With --gpus G each rank holds its own --voxels shard of one G*--voxels scene (weak scaling; --voxels 125000 --gpus 8 is
BASELINE config C4), or --scaling strong cuts ONE --voxels problem into G shards; the library all-reduces the lower
triangle of [H|g|r] with NCCL once per evaluation, and every multi-GPU run first checks a small sharded scene against
the same scene on one GPU ("mgpu_parity").

  value      : shard-iterations per second with the voxels already resident in HBM (G * K / t; strong: K / t)
  e2e        : the same through the host-buffer call, per call: balm_set_voxels from pinned host arrays + a 10-iteration
               damping_iter (the reference's cap) + poses back, copies inside the timed region
  roofline   : dominant kernel = the rank-3M symmetric update (SYRK, bavoxel.hpp:404-418 restated)
  cpu_baseline : the CPU oracle (port of the reference loop nest; Eigen/PCL/ROS are absent so the reference
               itself cannot be built here) timed on two bounded voxel samples of the same workload and extrapolated
               with slope + intercept

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--poses P --voxels M --precision fp64|tensor]
                  [--dump-outputs DIR]

--dump-outputs DIR writes what the last timed step returned as DIR/<name>.npy (float64). The inputs depend on the
arguments only, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the source tree may be read-only; the benchmark leaves nothing in it

PTS = 40
NOISE = 0.01
RANGE = 2.0
SEED = 10
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array of `arrays` as out_dir/<name>.npy in float64."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sus=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sus=1400.0, src="fallback")


class ClockSampler:
    """SM clock / throttle reasons DURING the timed region (B200_PROFILING.md recipe). Samples through NVML in a thread
    (first sample within milliseconds, so short runs are covered too); falls back to polling nvidia-smi."""

    def __init__(self, index):
        self.index = index
        self.rows = []      # (sm_mhz, sm_max_mhz, set of reasons[, board power in W])
        self.power_limit_w = None
        self.stop_flag = False
        self.thread = None
        self.proc = None

    def _nvml_loop(self, nv, h):
        bits = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        try:
            self.power_limit_w = nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
        except Exception:
            pass
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                try:
                    pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                except Exception:
                    pw = None
                self.rows.append((float(sm), float(mx), {k for k, b in bits.items() if r & b}, pw))
            except Exception:
                pass
            time.sleep(0.02)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[self.index]) if vis and vis.split(",")[self.index].isdigit() else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read_smi, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read_smi(self):
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(",")]
            if len(f) < 7:
                continue
            try:
                try:
                    pw = float(f[2])
                except ValueError:
                    pw = None
                self.rows.append((float(f[0]), float(f[1]),
                                  {n for n, v in zip(names, f[3:7]) if v.lower().startswith("active")}, pw))
            except ValueError:
                continue

    def mark(self):
        """Index of the next sample: rows[mark:] were taken after this call."""
        return len(self.rows)

    def stop(self, since=0):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        elif self.thread:
            self.thread.join(timeout=1)
        rows = self.rows[since:] or self.rows
        if not rows:
            return None
        reasons = set()
        for r in rows:
            reasons |= r[2]
        out = {"sm_mhz": float(np.median([r[0] for r in rows])), "sm_max_mhz": max(r[1] for r in rows),
               "reasons": sorted(reasons), "samples": len(rows)}
        pw = [r[3] for r in rows if len(r) > 3 and r[3] is not None]
        if pw:  # board power under load next to the enforced limit: the SYRK runs AT the limit (sw_power_cap)
            out["power_w"] = float(np.median(pw))
            out["power_limit_w"] = self.power_limit_w
        return out


def numpy_sample(n_poses, n_voxels, seed=SEED):
    """benchmark_virtual-shaped scene (benchmark_virtual.cpp:547-606, pose noise :491-503) generated with numpy only --
    the same construction as tests/scenes.py, vectorised over the poses of a plane. Keeps the reference arm free of any
    balm_b200 code. Every pose sees every plane: K = n_voxels * n_poses observations."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scenes
    rng = np.random.default_rng(seed)
    rot_end = rng.normal(-1, 1, 3)
    tra_end = rng.normal(-1, 1, 3)
    rot_end = rot_end / np.linalg.norm(rot_end) * 0.5
    tra_end = tra_end / np.linalg.norm(tra_end)
    Rs = np.stack([scenes.exp_so3(i / n_poses * rot_end) for i in range(n_poses)])
    ps = np.stack([i / n_poses * tra_end for i in range(n_poses)])
    obs = np.empty((n_voxels, n_poses, 10))
    for s in range(n_voxels):
        rot = scenes.exp_so3(rng.uniform(-np.pi, np.pi, 3))
        center = rng.uniform(-RANGE, RANGE, 3)
        loc = np.stack([rng.uniform(-0.5, 0.5, (n_poses, PTS)), rng.uniform(-0.5, 0.5, (n_poses, PTS)),
                        rng.normal(0, NOISE, (n_poses, PTS))], axis=2)
        w = loc @ rot.T + center
        b = np.einsum("jpk,jkl->jpl", w - ps[:, None, :], Rs)          # R_j^T (x - p_j)
        b = b.astype(np.float32).astype(np.float64)                     # PointXYZINormal stores floats
        P = np.einsum("jpa,jpb->jab", b, b)
        v = b.sum(1)
        obs[s, :, 0] = P[:, 0, 0]; obs[s, :, 1] = P[:, 0, 1]; obs[s, :, 2] = P[:, 0, 2]
        obs[s, :, 3] = P[:, 1, 1]; obs[s, :, 4] = P[:, 1, 2]; obs[s, :, 5] = P[:, 2, 2]
        obs[s, :, 6:9] = v
        obs[s, :, 9] = PTS
    row_ptr = np.arange(n_voxels + 1, dtype=np.int64) * n_poses
    pose_idx = np.tile(np.arange(n_poses, dtype=np.int32), n_voxels)
    coe = np.full(n_voxels, float(n_poses * PTS))
    Rn = [Rs[i] @ scenes.exp_so3(rng.normal(0, 2 / 57.3, 3) / 1.732) for i in range(n_poses)]
    pn = [ps[i] + rng.normal(0, 0.1, 3) / 1.732 for i in range(n_poses)]
    return row_ptr, pose_idx, obs.reshape(-1, 10), coe, scenes.pack_poses(Rn, pn)


class CpuArm:
    """The reference's CPU implementation of one LM iteration, timed on a BOUNDED sample of the workload.

    The reference (Eigen + PCL + ROS) cannot be built in this image, so this is the oracle port of its loop nest
    (oracle/balm_oracle.c): accumulation with 4 threads (bavoxel.hpp:1027), residual pass and pivoted LDL^T with one
    thread, gcc -O3 without -march=native (CMakeLists.txt:9). The O(M) passes are timed at TWO sample sizes and
    extrapolated with slope + intercept, so the O(n^2) work of an evaluation (four n x n memsets, the ordered reduce,
    the mirror) is counted once and not multiplied by M / sample; the n = 6N solve is timed at full size."""

    def __init__(self, n_poses, m_small, m_large, native=False):
        from oracle import oracle_py as orc
        self.N, self.m1, self.m2 = n_poses, m_small, m_large
        rp, pi, ob, co, init = numpy_sample(n_poses, m_large)
        self.init = init
        self.big = orc.Oracle(n_poses, rp, pi, ob, co, native=native)
        k1 = m_small * n_poses
        self.small = orc.Oracle(n_poses, rp[:m_small + 1], pi[:k1], ob[:k1], co[:m_small], native=native)

    def step(self, voxels_total, threads=4):
        """-> (seconds of this sample step, extrapolated seconds per LM iteration of the full workload, detail)"""
        t_begin = time.perf_counter()
        te, tr = [], []
        for o in (self.small, self.big):
            t0 = time.perf_counter()
            H, g, r = o.evaluate_threads(self.init, threads=threads)     # divide_thread_left (4) / the single-thread twin (1)
            te.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            o.residual(self.init)                                   # evaluate_only_residual, 1 thread
            tr.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        dx, trial, _ = self.big.lm_step(H, g, 0.01, self.init)      # (H + uD).ldlt().solve(-g) + update, 1 thread
        t_solve = time.perf_counter() - t0
        self.last = {"H": H, "g": g, "r": r, "dx": dx, "poses_trial": trial}   # of the larger sample
        dm = float(self.m2 - self.m1)
        se, sr = (te[1] - te[0]) / dm, (tr[1] - tr[0]) / dm          # seconds per voxel
        ie, ir = te[0] - se * self.m1, tr[0] - sr * self.m1          # per-evaluation O(n^2) overhead
        if ie < 0 or se <= 0:   # timing noise made the samples look super- or sub-linear: the proportional estimate
            se, ie = te[1] / self.m2, 0.0
        if ir < 0 or sr <= 0:
            sr, ir = tr[1] / self.m2, 0.0
        t_iter = (ie + se * voxels_total) + (ir + sr * voxels_total) + t_solve
        detail = {"t_eval_s": te, "t_residual_s": tr, "t_solve_s": t_solve, "eval_s_per_voxel": se,
                  "eval_intercept_s": ie, "residual_s_per_voxel": sr, "residual_intercept_s": ir,
                  "sample_voxels": [self.m1, self.m2]}
        return time.perf_counter() - t_begin, t_iter, detail

    def describe(self, voxels_total):
        return (f"{self.m1} and {self.m2} of {voxels_total} voxels at {self.N} poses; O(M) passes extrapolated with "
                f"slope + intercept from the two sizes; LDL^T n={6 * self.N} timed at full size; accumulation 4 threads "
                f"(bavoxel.hpp:1027), residual + LDL^T 1 thread; gcc -O3 without -march=native (CMakeLists.txt:9)")


def ref_headers_check(n_poses, m_small, port_eval_s):
    """The reference's OWN divide_thread_left (bavoxel.hpp:1025-1059, compiled from /root/reference's headers against
    stand-in Eigen into oracle/_ref/libbalm_ref.so, when that file travelled here) on the small sample, next to the port's
    time for the same call. A plausibility check of the port's speed, not a baseline: the stand-in has none of Eigen's
    vectorised kernels, and the reference leaks its per-observation `Co` blocks (bavoxel.hpp:312-320) -- which is why it
    runs in a process of its own: millions of small host allocations inside this one slowed the later e2e leg's
    balm_set_voxels from 8 ms to 1 s."""
    code = ("import sys, time, json; sys.path.insert(0, %r); import bench; from oracle import ref_py\n"
            "if not ref_py.available(): print('null'); sys.exit(0)\n"
            "rp, pi, ob, co, init = bench.numpy_sample(%d, %d)\n"
            "prob = ref_py.Problem(%d, rp, pi, ob)\n"
            "t0 = time.perf_counter(); prob.divide_thread_left(init)\n"
            "print(json.dumps({'t': time.perf_counter() - t0}))\n") % (ROOT, n_poses, m_small, n_poses)
    try:
        out = subprocess.run([sys.executable, "-B", "-c", code], capture_output=True, text=True, timeout=300)
        res = json.loads(out.stdout.strip().splitlines()[-1])
        if res is None:
            return None
        return {"ref_headers_standin_eigen_eval_s": res["t"], "port_eval_s": port_eval_s, "sample_voxels": m_small,
                "threads": 4}
    except Exception as e:  # the check must never take the bench down
        return {"error": str(e)[:120]}


def cpu_baseline_once(n_poses, voxels_total, m_small, m_large):
    arm = CpuArm(n_poses, m_small, m_large)
    _, t_iter, detail = arm.step(voxels_total)
    out = {"value": 1.0 / t_iter, "unit": "iter/s", "cores": 4, "kind": "port", "extrapolated": True,
           "sample": arm.describe(voxels_total), "detail": detail}
    chk = ref_headers_check(n_poses, m_small, detail["t_eval_s"][0])
    if chk:
        out["ref_headers_check"] = chk
    if n_poses * voxels_total <= 200000:  # C1: also the single-thread twin of benchmark_virtual.cpp:218-482 (SURVEY 8d)
        try:
            _, t_one, _ = arm.step(voxels_total, threads=1)
            out["value_single_thread_twin"] = 1.0 / t_one
        except Exception:
            pass
    try:  # labelled NON-reference column: the same port compiled with -march=native
        _, t_nat, _ = CpuArm(n_poses, m_small, m_large, native=True).step(voxels_total)
        out["value_march_native"] = 1.0 / t_nat
    except Exception:
        pass
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path. The reference needs Eigen, PCL and ROS,
    none of which exist in this image (no baseline/_ref; oracle/_ref holds the reference's headers compiled against
    stand-in Eigen, a correctness pin whose speed says nothing about Eigen's), so the arm times the oracle port of the
    reference loop nest (CpuArm). A step = one bounded sample of an LM iteration (both sample sizes + the full-size
    solve); `ms_per_step` is that measured time, `value` the throughput EXTRAPOLATED to the full workload from it.
    No balm_b200 code runs."""
    if rank != 0:
        return
    n, m = args.poses, args.voxels
    arm = CpuArm(n, args.cpu_sample_small, args.cpu_sample_large)
    wall, its, detail = [], [], None
    for i in range(args.warmup + args.steps):
        w, t, detail = arm.step(m)
        if i >= args.warmup:
            wall.append(w)
            its.append(t)
    t_iter = float(np.mean(its))
    val = 1.0 / t_iter
    if args.dump_outputs:
        out = dict(arm.last)
        H = out.pop("H")
        rows = np.sort(np.random.default_rng(SEED).choice(len(H), min(len(H), 64), replace=False))
        dump_outputs(args.dump_outputs, dict(out, H_rows=H[rows], H_row_index=rows))   # 64 seeded rows of the n x n H
    chk = ref_headers_check(n, args.cpu_sample_small, detail["t_eval_s"][0])  # once, outside the timed steps
    line = {
        "impl": "reference", "metric": "ba_iterations_per_sec", "value": val, "unit": "iter/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(wall)),
        "ms_per_iteration_extrapolated": 1e3 * t_iter, "extrapolated": True,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"BASELINE C3: BA LM iteration, {n} poses x {m} plane voxels (benchmark_virtual shape, "
                               f"{PTS} pts/obs), CPU oracle port of the reference loop nest; each step times a bounded "
                               f"sample and `value` is extrapolated to the full workload", "poses": n, "voxels": m},
        "cpu_baseline": {"value": val, "unit": "iter/s", "cores": 4, "kind": "port", "extrapolated": True,
                         "sample": arm.describe(m), "detail": detail},
        "e2e": {"value": val, "unit": "iter/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if chk:
        line["cpu_baseline"]["ref_headers_check"] = chk
    print(json.dumps(line), flush=True)


def mgpu_parity_check(rank, world, local_rank, prec, uid_bytes):
    """world > 1: a small fixed scene sharded over the ranks (the last rank's shard EMPTY when there are more ranks
    than needed, to exercise that path), evaluated and optimised through the NCCL path, against the same scene on rank
    0 alone. -> (ok, detail) on rank 0, (None, None) elsewhere."""
    import balm_b200
    from balm_b200 import shard
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import scenes
    sc = scenes.make_scene(n_poses=40, n_planes=400, seed=51, drop=0.2, pts_size=8)
    parts = shard.partition_voxels(sc["row_ptr"], world)
    c = balm_b200.Context(40, local_rank, prec)
    rp, pi, ob, co, _ = shard.shard_arrays(sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["coe"], None, *parts[rank])
    c.set_voxels(rp, pi, ob, co)
    c.comm_init(rank, world, uid_bytes)
    H, g, r = c.evaluate(sc["poses_init"])
    poses, tr, _ = c.damping_iter(sc["poses_init"], gauge_mode=2)      # default min_planes guard: a collective decision
    c.close()
    if rank != 0:
        return None, None
    c1 = balm_b200.Context(40, local_rank, prec)
    c1.set_voxels(sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["coe"])
    H1, g1, r1 = c1.evaluate(sc["poses_init"])
    p1, tr1, _ = c1.damping_iter(sc["poses_init"], gauge_mode=2)
    c1.close()
    eH = float(np.abs(H - H1).max() / np.abs(H1).max())
    eg = float(np.abs(g - g1).max() / np.abs(g1).max())
    er = float(abs(r - r1) / abs(r1))
    ep = float(np.abs(poses - p1).max())
    ok = bool(eH < (1e-12 if prec == 0 else 2e-8) and eg < 1e-12 and er < 1e-13 and ep < 1e-6 and len(tr) == len(tr1)
              and [t["accepted"] for t in tr] == [t["accepted"] for t in tr1])
    return ok, {"rel_H": eH, "rel_g": eg, "rel_r": er, "max_dpose": ep, "lm_iters": [len(tr), len(tr1)],
                "scene": "40 poses x 400 voxels, 20 % observations dropped, sharded by sum k^2"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="balm_b200")
    ap.add_argument("--poses", type=int, default=500)
    ap.add_argument("--voxels", type=int, default=100000,
                    help="plane voxels per GPU (weak scaling; 125000 x 8 GPUs = BASELINE C4) or in total (--scaling strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--precision", default=os.environ.get("BALM_BENCH_PRECISION", "tensor"), choices=["fp64", "tensor"])
    ap.add_argument("--cpu-sample-small", type=int, default=256)
    ap.add_argument("--cpu-sample-large", type=int, default=1024)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import balm_b200

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def new_uid():
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(balm_b200.Context.comm_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        return bytes(uid.cpu().numpy().tobytes())

    N = args.poses
    if args.scaling == "strong":  # one fixed problem of --voxels voxels, cut into `world` contiguous shards
        M_total = args.voxels
        first = rank * M_total // world
        M = (rank + 1) * M_total // world - first
    else:
        M, first, M_total = args.voxels, rank * args.voxels, world * args.voxels
    prec = balm_b200.PREC_TENSOR if args.precision == "tensor" else balm_b200.PREC_FP64

    mgpu_ok, mgpu_detail = None, None
    if world > 1:
        mgpu_ok, mgpu_detail = mgpu_parity_check(rank, world, local_rank, prec, new_uid())

    ctx = balm_b200.Context(N, local_rank, prec)
    gt, init = ctx.synth_virtual(M, first, PTS, NOISE, RANGE, SEED)
    if world > 1:
        ctx.comm_init(rank, world, new_uid())

    lm = dict(u0=0.01, v0=2.0, rel_tol=-1.0, gauge_mode=2, min_planes_per_pose=0, force_hess=True)

    # ---- HBM-resident timing ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    ctx.damping_iter(init, max_iter=args.warmup, **lm)
    ctx.reset_counters()
    barrier()
    mark = sampler.mark()
    ctx.timer_begin()
    poses, trace, _ = ctx.damping_iter(init, max_iter=args.steps, **lm)
    ms = ctx.timer_end()
    barrier()
    clocks = sampler.stop(mark)
    tm = ctx.timings()
    assert len(trace) == args.steps, (len(trace), args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {
            "poses": poses,   # N x 12 after the last timed step
            "lm_trace": [[t_[k_] for k_ in ("r1", "r2", "u", "v", "q", "q1", "accepted", "recomputed_hess", "not_pd")]
                         for t_ in trace]})
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    K = args.steps
    # weak: every rank advances its own shard (value counts shard-iterations, the unit the driver's efficiency is
    # computed in); strong: ONE problem, value = iterations of that problem per second
    value = (world if args.scaling == "weak" else 1) * K / (ms_max * 1e-3)

    # ---- end-to-end through the host-buffer call ----
    e2e = None
    if not args.no_e2e:
        row_ptr, pose_idx, obs10, coe = ctx.download_voxels()

        def pinned(a):
            tt = torch.from_numpy(a).pin_memory()
            return tt.numpy(), tt
        keep = []
        arrs = []
        for a in (row_ptr, pose_idx, obs10, coe):
            n_, t_ = pinned(a)
            arrs.append(n_)
            keep.append(t_)
        del row_ptr, pose_idx, obs10, coe
        h2d_call = sum(a.nbytes for a in arrs) + init.nbytes

        call_ms = []

        def timed_calls(iters_per_call, calls):
            """`calls` x [balm_set_voxels(pinned host arrays) + damping_iter(iters_per_call) + poses back]"""
            barrier()
            t0 = time.perf_counter()
            t_set = 0.0
            call_ms.clear()
            for _ in range(calls):
                ts = time.perf_counter()
                ctx.set_voxels(arrs[0], arrs[1], arrs[2], arrs[3])
                t_set += time.perf_counter() - ts
                p2, tr2, _ = ctx.damping_iter(init, max_iter=iters_per_call, **lm)   # returns with the poses on the host
                call_ms.append(1e3 * (time.perf_counter() - ts))
            ctx.sync()
            dt = time.perf_counter() - t0
            te = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            return float(te.item()), t_set / calls, p2

        timed_calls(1, 1)  # warms the allocator / page tables of the registration path
        # headline: one registration per damping_iter call of 10 iterations, the reference's own cap (bavoxel.hpp:1104)
        per_call = 10
        calls = max(1, (K + per_call - 1) // per_call)
        dt10, t_set10, p10 = timed_calls(per_call, calls)
        mult = world if args.scaling == "weak" else 1
        e2e = {"value": mult * per_call * calls / dt10, "unit": "iter/s",
               "h2d_bytes_per_step": int(h2d_call / per_call), "d2h_bytes_per_step": int(init.nbytes / per_call + 8 * 3),
               "iterations_per_call": per_call, "calls": calls, "set_voxels_ms": 1e3 * t_set10,
               "call_ms": [round(x, 2) for x in call_ms],  # the upload shares PCIe / host memory with the box's other tenants
               "value_best_call": mult * per_call / (1e-3 * min(call_ms)),
               "note": "per call: balm_set_voxels(pinned host CSR arrays, the whole voxel set) + damping_iter(10 "
                       "iterations = the reference's cap, bavoxel.hpp:1104) + poses back; the upload is amortised over "
                       "10 iterations only"}
        if K != per_call:  # the same with the upload amortised over all K steps (round 1's definition), for comparison
            dtk, t_setk, pk = timed_calls(K, 1)
            e2e["value_one_upload_for_all_steps"] = mult * K / dtk
            assert np.abs(pk - poses).max() < 1e-9  # same answer through the host path
        else:
            assert np.abs(p10 - poses).max() < 1e-9

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    n_eval = max(tm["n_eval"], 1)
    syrk_ms = tm["ms_syrk"] / n_eval
    k = N
    flops = 108.0 * k * (k + 1) * M  # SURVEY 8d: SYRK-half count per evaluation (this rank's shard)
    obs_bytes = 80.0 * M * N
    if args.precision == "tensor":
        peak_tf, peak_note = pk["bf16_sus"], f"bf16 dense sustained, {pk['src']} (int8 tcgen05 pipe is 2x bf16)"
    else:
        peak_tf, peak_note = pk["bf16_sus"], (f"bf16 dense sustained, {pk['src']}; the fp64 path runs on the DMMA "
                                              f"pipe whose nominal peak is 40 TFLOP/s (not in MEASURED_PEAKS.json)")
    ach_tf = flops / (syrk_ms * 1e-3) / 1e12
    # dram bytes per launch of the dominant kernel: NOT measurable inside this run (needs ncu); taken from the ncu
    # --set full capture of this same command committed under profiles/ for the CURRENT kernel, with its provenance,
    # or null when no capture matches this configuration
    traffic, traffic_src = None, None
    try:
        tr_ = json.load(open(os.path.join(ROOT, "profiles", "r2_syrk_traffic.json")))
        if (args.precision == "tensor" and tr_["poses"] == N and tr_["voxels"] == M):
            traffic, traffic_src = tr_["dram_bytes_per_launch"], tr_["source"]
    except Exception:
        pass
    roof = {"kernel": "syrk_f64_kernel" if args.precision == "fp64" else "syrk_tc_2sm_kernel", "bound": "tensor",
            "achieved": ach_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_tf / peak_tf, "traffic": traffic,
            "traffic_source": traffic_src,
            "peak_note": peak_note, "algorithmic_flops_per_launch": flops, "ms_per_launch": syrk_ms,
            "traffic_note": "algorithmic bytes of this kernel = digit planes read once (S x 3M x ldg B) + fp64 partial "
                            "tiles written"}
    if args.precision == "tensor":
        planes = tm["digit_planes"]
        pairs = planes * (planes + 1) // 2
        nbk = (6 * N + 127) // 128
        # 2-SM pairs: every tile once (tiles of consecutive even block columns are flipped to make every column's count
        # even); one duplicate slot only when the number of even columns is odd
        tiles_exec = nbk * (nbk + 1) // 2 + (((nbk + 1) // 2) % 2)
        int8_ops = 2.0 * pairs * tiles_exec * 128 * 128 * 3 * M
        roof["digit_planes"] = planes
        roof["executed_int8_tops"] = int8_ops / (syrk_ms * 1e-3) / 1e12
        roof["frac_int8"] = roof["executed_int8_tops"] / (2.0 * pk["bf16_sus"])
        roof["frac_int8_note"] = ("executed int8 digit-pair MMA rate against 2 x the measured bf16 SUSTAINED peak (the "
                                  "int8 tcgen05 pipe runs at twice the bf16 rate); `frac` above is the ALGORITHMIC fp64 "
                                  "flop rate against the bf16 sustained peak")
        roof["frac_of_int8_nominal_4500_tops"] = roof["executed_int8_tops"] / 4500.0
        roof["frac_of_2x_measured_bf16_burst"] = roof["executed_int8_tops"] / (2.0 * pk["bf16"])
    if args.precision == "fp64":
        roof["frac_of_fp64_nominal_40tf"] = ach_tf / 40.0
    res_ms = tm["ms_residual"] / max(tm["n_residual"], 1)
    stats_ms = tm["ms_stats"] / max(tm["n_stats"], 1) if tm["n_stats"] else res_ms
    obs_ms = tm["ms_obs"] / n_eval
    if args.precision == "tensor":
        gout = 18.0 * tm["digit_planes"]
        gnote = (f"80 B/obs read (counted once) + {gout:.0f} B/obs written (18 values x {tm['digit_planes']} int8 digit "
                 f"planes); {tm['single_sweeps']} of {n_eval} evaluations needed one sweep (scales speculated from the "
                 f"previous evaluation and accepted), {tm['redone_sweeps']} re-ran the digit sweep, the rest swept twice")
    else:
        gout, gnote = 144.0, "80 B/obs read + 144 B/obs fp64 G' written"
    hbm = {
        "residual_pass": {"bound": "hbm", "achieved": obs_bytes / (res_ms * 1e-3) / 1e9, "peak": pk["hbm"],
                          "unit": "GB/s", "frac": obs_bytes / (res_ms * 1e-3) / 1e9 / pk["hbm"], "ms": res_ms},
        "voxel_stats": {"bound": "hbm", "achieved": obs_bytes / (stats_ms * 1e-3) / 1e9, "peak": pk["hbm"],
                        "unit": "GB/s", "frac": obs_bytes / (stats_ms * 1e-3) / 1e9 / pk["hbm"], "ms": stats_ms,
                        "note": f"ran in {tm['n_stats']} of {n_eval} evaluations; the others took the eigen data "
                                f"from the residual pass of the accepted step (same kernel, same poses)"},
        "obs_pass": {"bound": "hbm", "achieved": (obs_bytes + gout * M * N) / (obs_ms * 1e-3) / 1e9,
                     "peak": pk["hbm"], "unit": "GB/s",
                     "frac": (obs_bytes + gout * M * N) / (obs_ms * 1e-3) / 1e9 / pk["hbm"], "ms": obs_ms,
                     "bytes_note": gnote},
    }
    phases = {k_: (tm[k_] / n_eval if k_ not in ("ms_solve", "ms_residual") else
                   tm[k_] / max(tm["n_solve" if k_ == "ms_solve" else "n_residual"], 1))
              for k_ in ("ms_stats", "ms_obs", "ms_slice", "ms_syrk", "ms_assemble", "ms_allreduce", "ms_solve",
                         "ms_residual")}

    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_baseline_once(N, M, args.cpu_sample_small, args.cpu_sample_large)

    cfg_name = ("BASELINE C4" if (N == 500 and M_total == 1000000) else "BASELINE C3" if (N == 500 and M == 100000)
                else "custom")
    line = {
        "metric": "ba_iterations_per_sec", "value": value, "unit": "iter/s", "n_gpus": world, "steps": K,
        "warmup": args.warmup, "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "f64" if args.precision == "fp64" else "s8 split-integer -> f64",
        "data": "synthetic",
        "config": {"workload": f"{cfg_name}: BA LM iteration, {N} poses x {M} plane voxels on this GPU "
                               f"({M_total} in the job), benchmark_virtual shape, {PTS} pts/obs, every pose sees every "
                               f"plane; " + ("value counts one iteration of each rank's shard (weak scaling)"
                                             if args.scaling == "weak" else
                                             "value counts iterations of the ONE job-wide problem (strong scaling)"),
                   "poses": N, "voxels_per_gpu": M, "total_voxels": M_total, "precision": args.precision,
                   "parallelism": f"voxel-shard x{world}, NCCL all-reduce of the upper triangle of [H|g|r] per evaluation",
                   "l2": "inputs (4.0 GB of observations per GPU) exceed the 126 MB L2; no explicit flush",
                   "lm": "force_hess=1, convergence exit disabled, 1 eval + 1 solve + 1 update + 1 residual per step"},
        "job_iter_per_s": K / (ms_max * 1e-3),
        "phases_ms": phases, "roofline": roof, "roofline_hbm": hbm, "cpu_baseline": cpu, "e2e": e2e,
        "gpu_launches": tm["launches"], "clocks": clocks,
        "sweeps": {"evaluations": tm["n_eval"], "stats_passes": tm["n_stats"], "single_sweeps": tm["single_sweeps"],
                   "redone_sweeps": tm["redone_sweeps"]},
        "lm_trace": [{"r1": t_["r1"], "r2": t_["r2"], "acc": t_["accepted"]} for t_ in trace[:4]],
    }
    if world > 1:
        line["mgpu_parity"] = mgpu_ok
        line["mgpu_parity_detail"] = mgpu_detail
        # the two serial terms that bound the scaling curve: both are per-iteration costs that do not shrink with the
        # number of GPUs (the all-reduce grows slowly with it; the solve is replicated on every rank)
        line["serial_terms_ms"] = {"allreduce": phases["ms_allreduce"], "replicated_solve": phases["ms_solve"]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
