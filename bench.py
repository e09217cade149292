#!/usr/bin/env python
"""bench.py -- faces/sec through data costs + MRF view selection + global seam leveling.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line
on rank 0.  A "step" is one pass of the hot path over the synthetic workload:
    value  : inputs already resident in HBM (mesh, images, graph uploaded before the timed region)
    e2e    : the three reference-facing C-ABI calls with HOST (pinned) buffers, H2D/D2H inside the
             timed region (b2tex_calculate_data_costs -> b2tex_view_selection ->
             b2tex_global_seam_leveling; what a texrecon drop-in does)
    roofline    : dominant kernel group of the step, CUDA-event time measured live (library events on
                  the launching stream), algorithmic bytes per DESIGN.md section 4
    cpu_baseline: the oracle (CPU restatement, kind "port") on a bounded sample of the same workload
`--impl reference` times the oracle port on the host cores (the reference itself is unbuildable
offline: MVE/rayint/Eigen/mapMAP absent, SURVEY.md 0.2).
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "faces/sec (data-cost + MRF label + seam-level)"
UNIT = "faces/s"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_workload(scene_mod, name):
    t = time.time()
    s = scene_mod.config(name)
    ap, ai = scene_mod.face_adjacency(s.faces)
    rings = scene_mod.vertex_rings(s.faces, s.verts.shape[0])
    return s, (ap, ai), rings, time.time() - t


def workload_config(name, s, world):
    """The `config` object of the JSON line: a pure function of the workload and the GPU count, so that the two arms
    (`--impl b200` / `--impl reference`) print the same object; run-dependent numbers go under `run`."""
    par = importlib.import_module("mvs-texturing_b200.sharded")
    kind = {"C3": ", displaced icosphere", "C2": ", value-noise terrain", "C5": ", value-noise terrain"}.get(name, "")
    return {"workload": f"{name}: {s.num_faces} faces / {s.num_views} views {s.width}x{s.height}{kind}",
            "parallelism": par.describe_parallelism(world),
            "l2": f"inputs larger than L2 (images {s.images.nbytes / 1e9:.2f} GB, data costs ~{10 * 44 * s.num_faces / 1e9:.1f} GB)"
                  if s.images.nbytes > 256e6 else "L2 flushed by the data-cost stage itself (every step re-reads all images)"}


# --------------------------------------------------------------------------------------------------
# CPU baseline: oracle port on a bounded sample (first `fs` faces; occlusion against the whole mesh)
# --------------------------------------------------------------------------------------------------
def cpu_sample(scene_mod, s, fs, threads):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    fs = min(fs, s.num_faces)
    t0 = time.time()
    dc = O.data_costs(s, threads=threads, face_range=(0, fs))
    t1 = time.time()
    sub_faces = s.faces[:fs]
    used, inv = np.unique(sub_faces.ravel(), return_inverse=True)
    f2 = inv.reshape(-1, 3).astype(np.uint32)
    sub = scene_mod.Scene(np.ascontiguousarray(s.verts[used]), f2, s.face_normals[:fs], s.pos, s.viewdir,
                          s.proj, s.w2c, s.width, s.height, s.images, "sample")
    ap, ai = scene_mod.face_adjacency(f2)
    rings = scene_mod.vertex_rings(f2, len(used))
    fp = dc["face_ptr"][:fs + 1].copy()
    t2 = time.time()
    m = O.view_selection(ap, ai, fp, dc["view"], dc["cost"], threads=threads)
    t3 = time.time()
    g = O.global_seam_leveling(sub, rings, m["labels"])
    t4 = time.time()
    tt = (t1 - t0) + (t3 - t2) + (t4 - t3)
    return dict(faces=fs, seconds=tt, dc_s=t1 - t0, mrf_s=t3 - t2, seam_s=t4 - t3, value=fs / tt,
                mrf_energy=m["energy"], mrf_iterations=m["iterations"], cg_iterations=g["iterations"])


def run_reference(args, rank, world):
    """Reference arm: the CPU implementation of the path (oracle port: stock texrecon is unbuildable offline) on the host
    cores, same `config` object as the b200 arm, each step a bounded sample of that workload (cpu_baseline.sample)."""
    if rank != 0:
        return
    scene_mod = importlib.import_module("mvs-texturing_b200.scene")
    s = scene_mod.config(args.workload)
    cores = os.cpu_count() or 1
    fs = args.cpu_faces or max(2000, min(s.num_faces, int(2.0e9 / max(1, s.num_views) / 100)))
    times, last = [], None
    for i in range(args.warmup + args.steps):
        r = cpu_sample(scene_mod, s, fs, cores)
        if i >= args.warmup:
            times.append(r["seconds"])
        last = r
    t = statistics.median(times)
    val = fs / t
    # is the per-face rate of the sample the rate of a larger piece of the same workload?  (one extra run at 4x the faces)
    rate_check = None
    if fs * 4 <= s.num_faces and not args.no_rate_check:
        r4 = cpu_sample(scene_mod, s, fs * 4, cores)
        rate_check = {"faces": [fs, fs * 4], "faces_per_s": [val, r4["value"]]}
    out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(args.workload, s, args.gpus),
           "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                            "sample": f"oracle (CPU restatement; stock texrecon is unbuildable offline) on the first {fs} of "
                                      f"{s.num_faces} faces x all {s.num_views} views per step, occlusion against the whole "
                                      f"mesh; median of {len(times)} steps (min {fs / max(times):.0f}, max {fs / min(times):.0f} "
                                      f"faces/s); last step dc {last['dc_s']:.2f}s mrf {last['mrf_s']:.2f}s seam {last['seam_s']:.2f}s",
                            "rate_check": rate_check},
           "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------------------
# parity at the benchmarked size: the oracle on the WHOLE workload against what the timed run left on the device
# --------------------------------------------------------------------------------------------------
def verify_against_oracle(scene_mod, s, adj, rings, runner, res, world):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import zlib
    import oracle as O
    cores = os.cpu_count() or 1
    c = runner.ctx
    t0 = time.time()
    o = O.data_costs(s, threads=cores)
    t1 = time.time()
    om = O.view_selection(adj[0], adj[1], o["face_ptr"], o["view"], o["cost"], threads=cores, num_parts=world)
    t2 = time.time()
    og = O.global_seam_leveling(s, rings, om["labels"])
    t3 = time.time()
    out = {"oracle_seconds": {"data_costs": round(t1 - t0, 2), "view_selection": round(t2 - t1, 2), "seam_leveling": round(t3 - t2, 2)},
           "oracle_cores": cores, "num_parts": world}
    crc = lambda a: zlib.crc32(np.ascontiguousarray(a).tobytes())
    if world == 1:
        dc = c.data_costs_download(int(res["dc"].nnz))
        out["data_costs_bit_exact"] = bool(len(dc["view"]) == len(o["view"]) and np.array_equal(dc["face_ptr"], o["face_ptr"])
                                           and np.array_equal(dc["view"], o["view"])
                                           and np.array_equal(dc["cost"].view(np.uint32), o["cost"].view(np.uint32)))
        out["crc_data_costs"] = [crc(dc["face_ptr"]), crc(dc["view"]), crc(dc["cost"])]
        out["crc_data_costs_ref"] = [crc(o["face_ptr"]), crc(o["view"]), crc(o["cost"])]
    labels = c.labels_download()
    out["labels_bit_exact"] = bool(np.array_equal(labels, om["labels"]))
    out["crc_labels"], out["crc_labels_ref"] = crc(labels), crc(om["labels"])
    out["mrf_iterations_ref"] = int(om["iterations"])
    out["mrf_energy_ref"] = float(om["energy"])
    out["mrf_energy_fixed_ref"] = int(O.mrf_energy_fixed(adj[0], adj[1], o["face_ptr"], o["view"], o["cost"], om["labels"]))
    out["mrf_energy_fixed"] = int(round(res["mrf"].energy_final * 4294967296.0))
    out["mrf_energy_identical"] = out["mrf_energy_fixed"] == out["mrf_energy_fixed_ref"]
    x = c.seam_download(res["seam"])["x"]
    out["seam_rows_equal"] = bool(int(res["seam"].num_rows) == len(og["row_label"]))
    seam_ok = False
    if out["seam_rows_equal"] and out["labels_bit_exact"]:
        import scipy.sparse as sp
        cp, cc, cv = og["csr"]
        A = sp.csr_matrix((cv.astype(np.float64), cc.astype(np.int64), cp.astype(np.int64)), shape=(len(cp) - 1,) * 2)
        x64, rhs = x.astype(np.float64), og["rhs"].astype(np.float64)
        # north_star's bar: the residual of the returned adjust values on the reference system, relative L2, per channel
        out["seam_true_residual"] = [float(np.linalg.norm(A @ x64[:, ch] - rhs[:, ch]) / max(1e-300, np.linalg.norm(rhs[:, ch])))
                                     for ch in range(3)]
        out["seam_true_residual_ref"] = [float(np.linalg.norm(A @ og["x"][:, ch].astype(np.float64) - rhs[:, ch]) /
                                               max(1e-300, np.linalg.norm(rhs[:, ch]))) for ch in range(3)]
        out["seam_rel_l2_vs_ref"] = float(np.linalg.norm(x - og["x"]) / max(1e-30, np.linalg.norm(og["x"])))
        out["cg_iterations_ref"] = [int(v) for v in og["iterations"]]
        same_stop = list(res["seam"].iterations) == out["cg_iterations_ref"]
        # the system is singular and the residual hovers around 1e-4 for ~20 iterations while x still moves ~0.25 % per
        # iteration (measured on C3, NOTES.md): the distance of the solutions is only meaningful for equal stop iterations
        out["seam_same_stop_iterations"] = bool(same_stop)
        seam_ok = max(out["seam_true_residual"]) < 2e-4 and out["seam_rel_l2_vs_ref"] < (5e-3 if same_stop else 5e-2)
    out["ok"] = bool(out["labels_bit_exact"] and out["mrf_energy_identical"] and out.get("data_costs_bit_exact", True) and seam_ok)
    out["cpu_full_workload"] = {"value": s.num_faces / (t3 - t0), "unit": UNIT, "seconds": round(t3 - t0, 2)}
    return out


# --------------------------------------------------------------------------------------------------
# outputs of the timed path, for comparing two builds of the project output for output
# --------------------------------------------------------------------------------------------------
DUMP_ROWS = 1 << 18   # at most 7 arrays of 2^18 rows (+ their row positions): about 35 MB per dump


def dump_outputs(directory, arrays):
    """Writes every array as <directory>/<name>.npy, integers as float64 (exact) and floats as float32.  An array with more
    than DUMP_ROWS rows is replaced by a seeded sample of its rows (the same positions for the same length in every run);
    the positions go to <name>.rows.npy."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        if len(a) > DUMP_ROWS:
            rows = np.sort(np.random.default_rng(0).choice(len(a), DUMP_ROWS, replace=False))
            np.save(os.path.join(directory, f"{name}.rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(directory, f"{name}.npy"), a.astype(np.float64 if a.dtype.kind in "iu" else np.float32))


def timed_path_outputs(runner, res, world):
    """What a caller of the resident path receives after a step: data costs (one GPU: the whole CSR), labels, adjust values."""
    c = runner.ctx
    out = {}
    if world == 1:
        dc = c.data_costs_download(int(res["dc"].nnz))
        out.update(data_costs_face_ptr=dc["face_ptr"], data_costs_view=dc["view"], data_costs_cost=dc["cost"])
    out["labels"] = c.labels_download()
    seam = c.seam_download(res["seam"])
    out.update(seam_row_ptr=seam["row_ptr"], seam_row_label=seam["row_label"], seam_x=seam["x"])
    return out


# --------------------------------------------------------------------------------------------------
def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--gpus", type=int, default=1)
    ap_.add_argument("--steps", type=int, default=5)
    ap_.add_argument("--warmup", type=int, default=3)
    ap_.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap_.add_argument("--workload", default="C3")
    ap_.add_argument("--cpu-faces", type=int, default=0, help="faces in the CPU baseline sample (0 = auto)")
    ap_.add_argument("--no-cpu-baseline", action="store_true")
    ap_.add_argument("--no-rate-check", action="store_true")
    ap_.add_argument("--no-e2e", action="store_true")
    ap_.add_argument("--no-verify", action="store_true",
                     help="skip the parity check of the timed run's results against the oracle on the whole workload "
                          "(about a minute of CPU time on rank 0)")
    ap_.add_argument("--with-patches", action="store_true",
                     help="also time texture patches + adjust_colors + local seam leveling (reported under 'extra_stages'; "
                          "never part of the headline metric, which is the three north_star stages)")
    ap_.add_argument("--dump-outputs", metavar="DIR",
                     help="write what the last timed step computed (data costs, labels, adjust values) as DIR/<name>.npy; "
                          "arrays longer than 2^18 rows as a fixed seeded sample of rows; on several GPUs without the data "
                          "costs, which stay split over the ranks (--impl b200 only)")
    args = ap_.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap_.error("--dump-outputs writes the results of the timed GPU path: use it with --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank, world)

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    b2 = importlib.import_module("mvs-texturing_b200")
    scene_mod = importlib.import_module("mvs-texturing_b200.scene")
    par = importlib.import_module("mvs-texturing_b200.sharded")

    s, (ap, ai), rings, gen_s = build_workload(scene_mod, args.workload)
    F, K = s.num_faces, s.num_views
    hbm_peak, peak_src = peaks()

    # ---- resident arm ---------------------------------------------------------------------------
    runner = par.ShardedPipeline(b2, s, (ap, ai), rings, rank, world, local_rank)
    ext = torch.cuda.ExternalStream(runner.ctx.stream(), device=torch.device("cuda", local_rank))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        res = runner.step()
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    runner.ctx.profile(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = runner.ctx.launch_count()
    t0 = time.perf_counter()
    ev0.record(ext)
    for _ in range(args.steps):
        res = runner.step()
    ev1.record(ext)
    sync_all()
    wall = time.perf_counter() - t0
    launches = runner.ctx.launch_count() - l0
    dev_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    prof = runner.ctx.profile_report()
    runner.ctx.profile(False)
    t_local = torch.tensor([dev_ms / 1e3], dtype=torch.float64, device="cuda")
    n_launch = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
        dist.all_reduce(n_launch)
    t_total = float(t_local.item())
    ms_per_step = 1e3 * t_total / args.steps
    value = F / (t_total / args.steps)
    total_nnz = runner.total_nnz() or int(res["dc"].nnz)

    # per kernel-group aggregation (this rank); launch groups that ran after the stop rule fired are no-ops (< 2 us)
    agg = {}
    for name, ms, by in prof:
        a = agg.setdefault(name, [0, 0.0, 0.0])
        a[0] += 1; a[1] += ms; a[2] += by
    kernels = [{"name": n, "launch_groups": c, "ms_per_step": ms / args.steps, "algorithmic_mb_per_step": by / args.steps / 1e6,
                "gbs": (by / ms / 1e6) if ms > 0 else 0.0} for n, (c, ms, by) in agg.items()]
    # the PCG kernel is timed by its own events inside seam_run
    pcg_ms = res["seam"].cg_ms
    R, nnzL, its = res["seam"].num_rows, res["seam"].nnz_full, res["seam"].cg_launch_iterations
    # SURVEY 8d formula with the storage actually used: 4 B per Laplacian entry (column | weight class)
    # + 4 B diagonal value per row instead of 8 B (value + column) per entry; rows of this rank only
    pcg_bytes = its * (4.0 * nnzL + 4.0 * R + 4.0 * (R + 1) + 13 * 4.0 * R * 3) / world
    kernels.append({"name": "k_pcg" if world == 1 else "k_pcg_mg", "launch_groups": 1, "ms_per_step": pcg_ms,
                    "algorithmic_mb_per_step": pcg_bytes / 1e6, "gbs": pcg_bytes / pcg_ms / 1e6 if pcg_ms else 0.0, "iterations": its})
    kernels.sort(key=lambda k: -k["ms_per_step"])
    dom = kernels[0]
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")  # dram bytes/launch from the committed ncu captures
    if os.path.exists(tp) and args.workload == "C3" and world == 1:
        key = dom["name"].replace("mrf.", "").replace("dc.", "").split("+")[0].split("<")[0]
        traffic = json.load(open(tp)).get(key)
    mrf_it = int(res["mrf"].iterations)
    per_step_launches = {"k_pcg": 1, "k_pcg_mg": 1}.get(dom["name"], mrf_it if dom["name"].startswith("mrf.") else 1)
    roofline = {"kernel": dom["name"], "bound": "hbm", "achieved": dom["gbs"], "peak": hbm_peak, "unit": "GB/s",
                "frac": dom["gbs"] / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "launches_per_step": per_step_launches, "ms_per_launch": dom["ms_per_step"] / per_step_launches,
                "algorithmic_bytes_per_launch": dom["algorithmic_mb_per_step"] * 1e6 / per_step_launches,
                "note": "algorithmic bytes per DESIGN.md section 4 (SURVEY 8d); traffic = dram bytes of one "
                        "launch from the ncu --set full capture summarised in profiles/ (C3 workload)"}
    stage_ms = {k: 1e3 * v / 1 for k, v in res["stage_s"].items()}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, timed_path_outputs(runner, res, world))

    # ---- parity of the timed run's results at the benchmarked size ---------------------------------
    verify = None
    if not args.no_verify and rank == 0:
        verify = verify_against_oracle(scene_mod, s, (ap, ai), rings, runner, res, world)
    sync_all()

    # ---- e2e arm: the reference-facing C-ABI call(s) with HOST buffers --------------------------------
    e2e = None
    if not args.no_e2e and rank == 0 and world == 1:
        e2e = par.e2e_host_path(b2, torch, s, (ap, ai), rings, steps=max(1, min(args.steps, 5)), warmup=2)
    elif not args.no_e2e:
        e2e = runner.e2e(torch, steps=max(1, min(args.steps, 3)), warmup=1)
    sync_all()

    extra = None
    if args.with_patches and rank == 0 and world == 1:
        # after the timed region, on the labels / offsets the last step left on the device
        ctx = runner.ctx
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        torch.cuda.synchronize()
        ev[0].record(ext)
        pinfo = ctx.texture_patches_run(apply_adjust=True)
        ev[1].record(ext)
        linfo = ctx.local_seam_leveling_run()
        ev[2].record(ext)
        torch.cuda.synchronize()
        extra = {"texture_patches_ms": ev[0].elapsed_time(ev[1]), "local_seam_leveling_ms": ev[1].elapsed_time(ev[2]),
                 "patches": int(pinfo.num_patches), "patch_pixels": int(pinfo.num_pixels), "seam_edges": int(linfo.num_seam_edges),
                 "poisson_unknowns": int(linfo.num_unknowns), "poisson_iterations": list(linfo.iterations),
                 "note": "includes the host bookkeeping (component BFS, merge plan, seam edges) inside each call"}

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        fs = args.cpu_faces or max(2000, min(F, int(2.0e9 / max(1, K) / 100)))
        r = cpu_sample(scene_mod, s, fs, cores)
        cpu = {"value": r["value"], "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"oracle (CPU restatement, NOT stock texrecon) on the first {fs} of {F} faces x all {K} "
                         f"views, occlusion against the whole mesh: {r['seconds']:.1f}s "
                         f"(dc {r['dc_s']:.1f} mrf {r['mrf_s']:.1f} seam {r['seam_s']:.1f})"}
        # like for like: the GPU path on the identical sub-mesh
        cpu["gpu_same_sample"] = gpu_same_sample(b2, scene_mod, s, fs)
        if verify:
            cpu["whole_workload"] = verify["cpu_full_workload"]

    if rank == 0:
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": workload_config(args.workload, s, world),
               "run": {"nnz": int(total_nnz), "mrf_iterations": mrf_it, "mrf_energy": res["mrf"].energy_final,
                       "mrf_energy_ref": verify["mrf_energy_ref"] if verify else None,
                       "cg_iterations": list(res["seam"].iterations), "cg_residual": [float(x) for x in res["seam"].residual],
                       "scene_setup_s": round(gen_s, 1),
                       "device_memory_in_use_gb": round((lambda fr, tot: (tot - fr) / 1e9)(*torch.cuda.mem_get_info()), 2)},
               "stage_ms": stage_ms, "kernels": kernels[:10], "roofline": roofline, "cpu_baseline": cpu,
               "verify": verify, "e2e": e2e, "extra_stages": extra, "gpu_launches": int(n_launch.item()), "clocks": clocks,
               "wall_ms_per_step": 1e3 * wall / args.steps}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def gpu_same_sample(b2, scene_mod, s, fs):
    """The resident GPU pipeline on the sub-mesh the CPU sample uses (first fs faces, all views)."""
    fs = min(fs, s.num_faces)
    sub_faces = s.faces[:fs]
    used, inv = np.unique(sub_faces.ravel(), return_inverse=True)
    f2 = inv.reshape(-1, 3).astype(np.uint32)
    sub = scene_mod.Scene(np.ascontiguousarray(s.verts[used]), f2, np.ascontiguousarray(s.face_normals[:fs]), s.pos, s.viewdir,
                          s.proj, s.w2c, s.width, s.height, s.images, "sample")
    adj = scene_mod.face_adjacency(f2)
    rings = scene_mod.vertex_rings(f2, len(used))
    c = b2.Context(0)
    try:
        c.set_scene(sub); c.set_adjacency(*adj); c.set_vertex_rings(*rings)
        best = None
        for _ in range(3):
            c.synchronize()
            t0 = time.perf_counter()
            c.data_costs_run(); c.view_selection_run(); c.seam_run()
            c.synchronize()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    finally:
        c.close()
    return {"value": fs / best, "unit": UNIT, "ms": 1e3 * best,
            "note": "occlusion against the sub-mesh only (the CPU sample traces against the whole mesh)"}


if __name__ == "__main__":
    main()
