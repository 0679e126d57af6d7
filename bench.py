#!/usr/bin/env python
"""Benchmark of the iALS hot path (BASELINE.json metric: iALS epochs/sec &
interactions/sec at k=128).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one iALS epoch (Gram(item) -> solve users -> Gram(user) -> solve
items) over a synthetic interaction matrix.  N=1 runs BASELINE.json configs[1]
(ML-20M shape 138493 x 26744, 20.0M nnz, K=128, CG with 3 steps) and, beside it
(key `c4_single_gpu`), the 1 B-interaction matrix of configs[3] on the one GPU --
the strong-scaling reference of the N>1 lines.  N>1 (under torch.distributed.run)
runs configs[3]: the 10M x 2M, 1 B-interaction power-law matrix row-sharded over
the N GPUs (strong scaling), plus the configs[4] top-100 sample.  One JSON
line is printed by rank 0 (see DESIGN.md "Measurement" for every field).

  value     whole-job interactions/s with the matrix and factors resident in HBM
            (CUDA events on the launching stream around exactly K epochs).
  e2e       the same metric through the reference-facing API with HOST buffers:
            every step uploads both factor matrices from pinned host memory,
            runs IALSTrainer.step() and reads both matrices back.
  roofline  the CG row-solve kernel (dominant): algorithmic bytes per launch /
            its CUDA-event duration vs the measured HBM peak.
  cpu_baseline  the CPU oracle (a port of the reference's C++/Eigen trainer,
            oracle/) on this box's host cores, same matrix, same factors.

`--impl reference` times that CPU port alone with all host threads (the real
irspack cannot be built offline: Eigen 5.0.1 / nanobind are not in the image).

`--dump-outputs DIR` (N=1 only) writes the factors the timed epochs produced (after
the last one) to DIR/<name>.npy, so that two builds can be compared output for
output: the inputs are seeded and identical for identical arguments.  The sharded
N>1 run keeps each rank's factor rows on its own GPU and has no such dump.
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

import numpy as np  # noqa: E402

METRIC = "ials_interactions_per_sec_k128"
UNIT = "interactions/s"
HYPER = dict(alpha0=0.1, reg=1e-3, nu=1.0, max_cg_steps=3)  # SURVEY.md 8 d


def oracle_row_check(before, after, other, rows, solver, hyper):
    """Parity at full size inside the bench (irspack_b200.dist.run_c4's ``parity_check``): the sampled
    rows of one more user half-epoch are re-solved by the CPU oracle (test infrastructure, here as
    the checker only) from the same inputs -- the other side's factors, their Gram, the rows' own
    previous values -- and compared with what the GPU wrote."""
    import numpy as np

    import oracle

    nt = oracle.hardware_threads()
    P = oracle.gram(other, hyper["alpha0"], nt)
    tgt = before.copy()
    if solver == "CG":
        oracle.step_cg(tgt, rows, other, P, hyper["alpha0"], hyper["reg"], hyper["nu"], oracle.LOSS_IALSPP,
                       hyper["max_cg_steps"], nt)
    else:
        oracle.step_cholesky(tgt, rows, other, P, hyper["alpha0"], hyper["reg"], hyper["nu"], oracle.LOSS_IALSPP, nt)
    err = float(np.abs(after - tgt).max() / (np.abs(tgt).max() + 1e-30))
    return {"rows": int(rows.shape[0]), "longest_row": int(np.diff(rows.indptr).max()),
            "max_abs_diff_over_max_abs_oracle": err, "tolerance": 2e-4, "ok": bool(err <= 2e-4),
            "what": "one more user half-epoch on all ranks; rank 0's sampled rows (random + its longest) "
                    "re-solved by the CPU oracle (float32 port) from the same item factors, Gram and "
                    "previous row values"}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured"
    return 6650.0, "fallback"  # /opt/skills/guides/B200_PROFILING.md


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "25", "-i", str(self.device)], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)),
                "reasons": sorted(reasons), "samples": len(sm)}


def workload(n_gpus: int):
    from irspack_b200.synth import SHAPES

    U, I, nnz, K = SHAPES["ml20m"]
    return dict(name="ml20m", n_users=U, n_items=I, nnz=nnz, K=K, seed=1002)


def make_inputs(w):
    from irspack_b200.synth import init_factors, synth_csr

    X = synth_csr(w["n_users"], w["n_items"], w["nnz"], seed=w["seed"])
    return X, init_factors(w["n_users"], w["K"], 1), init_factors(w["n_items"], w["K"], 2)


DUMP_USER_ROWS = 65536  # all 138493 user rows (71 MB) and the item factors would exceed the 64 MB dump budget


def dump_outputs(out_dir, user, item):
    """What a caller of the timed path receives after its last epoch: the item factors whole and a
    fixed, seeded sample of user rows (ascending), float32."""
    os.makedirs(out_dir, exist_ok=True)
    n = user.shape[0]
    rows = np.sort(np.random.default_rng(0).choice(n, min(n, DUMP_USER_ROWS), replace=False))
    np.save(os.path.join(out_dir, "user_factors_sample.npy"), np.ascontiguousarray(user[rows], dtype=np.float32))
    np.save(os.path.join(out_dir, "item_factors.npy"), np.ascontiguousarray(item, dtype=np.float32))


def solve_bytes(w):
    """Algorithmic bytes of the two row-solve launches of one epoch (DESIGN.md):
    every neighbour's K-vector + int32 index + f32 value once per half-epoch,
    own row read + written, indptr."""
    U, I, nnz, K = w["n_users"], w["n_items"], w["nnz"], w["K"]
    return 2 * nnz * (4 * K + 8) + (U + I) * 8 * K + (U + I + 2) * 8


def epoch_bytes(w):  # SURVEY.md 8 d, B_cg (adds the Gram's read of each factor matrix)
    return solve_bytes(w) + (w["n_users"] + w["n_items"]) * 4 * w["K"]


def cpu_epochs(w, X, u0, i0, n_epochs, n_threads):
    """Seconds per epoch of the CPU port (oracle) on this host."""
    import oracle

    if n_epochs <= 0:  # A/B runs (tools/gpu_ab.sh) skip the CPU leg
        return [float("nan")]
    o = oracle.OracleTrainer(X, w["K"], HYPER["alpha0"], HYPER["reg"], HYPER["nu"],
                             oracle.LOSS_IALSPP)
    o.user, o.item = u0.copy(), i0.copy()
    o.epoch_native(oracle.SOLVER_CG, HYPER["max_cg_steps"], n_threads)  # warm-up (page-in, caches)
    times = []
    for _ in range(n_epochs):
        t = time.perf_counter()
        o.epoch_native(oracle.SOLVER_CG, HYPER["max_cg_steps"], n_threads)
        times.append(time.perf_counter() - t)
    return times


C4_CPU_SAMPLE_SCALE = 0.01  # the reference arm's bounded sample of configs[3]: 100k x 20k, 10 M nnz


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle

    if args.gpus > 1:
        # configs[3] does not fit a CPU run of minutes (1 B interactions ~ 25 s per epoch per
        # 40 M interactions/s): interactions/s is a rate, so the bounded sample is the same
        # power-law generator at 1 % of the shape
        from irspack_b200.dist import c4_shape
        from irspack_b200.synth import init_factors, synth_csr

        U, I, nnz, K = c4_shape(C4_CPU_SAMPLE_SCALE, 1)
        w = dict(name="powerlaw1b sample", n_users=U, n_items=I, nnz=nnz, K=K, seed=1004)
        X = synth_csr(U, I, nnz, seed=1004)
        u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
        sample = (f"{args.steps} full epochs of a {C4_CPU_SAMPLE_SCALE:.0%} sample of configs[3] (same power-law "
                  f"generator: {U}x{I}, {nnz} of 1e9 interactions); interactions/s is a rate")
    else:
        w = workload(args.gpus)
        X, u0, i0 = make_inputs(w)
        sample = f"{args.steps} full epochs of the whole workload"
    nt = oracle.hardware_threads()
    o = oracle.OracleTrainer(X, w["K"], HYPER["alpha0"], HYPER["reg"], HYPER["nu"],
                             oracle.LOSS_IALSPP)
    o.user, o.item = u0.copy(), i0.copy()
    for _ in range(args.warmup):
        o.epoch_native(oracle.SOLVER_CG, HYPER["max_cg_steps"], nt)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        o.epoch_native(oracle.SOLVER_CG, HYPER["max_cg_steps"], nt)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, o.user, o.item)
    value = w["nnz"] * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "epochs_per_sec": args.steps / dt,
        "config": config_dict(w, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nt, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def config_dict(w, n_gpus):
    if n_gpus > 1:
        return sharded_config_dict(n_gpus)
    return {
        "workload": f"iALS epoch, synthetic ML-20M shape {w['n_users']}x{w['n_items']}, "
                    f"{w['nnz']} nnz, K={w['K']}, CG max_cg_steps={HYPER['max_cg_steps']}, "
                    f"alpha0={HYPER['alpha0']}, reg={HYPER['reg']}, loss_type=IALSPP",
        "n_users": w["n_users"], "n_items": w["n_items"], "nnz": w["nnz"], "K": w["K"],
        "solver": "CG", "parallelism": "single GPU",
        "l2": "per-epoch working set (CSR + CSR^T 0.48 GB + factors 0.085 GB) exceeds the "
              "126 MB L2; no explicit flush",
    }


def sharded_config_dict(world):
    """`config` of the N > 1 run (irspack_b200/dist.py bench_main): BASELINE configs[3], the
    1 B-interaction power-law matrix row-sharded over the N GPUs.  Shared by both arms."""
    from irspack_b200.dist import c4_config_dict

    return c4_config_dict(world, float(os.environ.get("IALS_BENCH_C4_SCALE", "1.0")))


def run_ours(args):
    import torch

    import irspack_b200
    from irspack_b200 import _ials_core as core

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    if not torch.cuda.is_available() or irspack_b200.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device: irspack_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        from irspack_b200 import dist as ials_dist

        return ials_dist.bench_main(args, METRIC, UNIT, HYPER, parity_check=oracle_row_check)

    w = workload(1)
    X, u0, i0 = make_inputs(w)
    cfg = (core.IALSModelConfigBuilder().set_K(w["K"]).set_alpha0(HYPER["alpha0"])
           .set_reg(HYPER["reg"]).set_nu(HYPER["nu"]).build())
    sc = core.IALSSolverConfigBuilder().set_max_cg_steps(HYPER["max_cg_steps"]).build()
    tr = core.IALSTrainer(cfg, X)
    tr.user, tr.item = u0, i0
    launch_count = irspack_b200._lib.lib.ials_kernel_launch_count

    # ---- device-resident throughput ----
    for _ in range(args.warmup):
        tr.step_async(sc)
    tr.sync()
    tr.set_profiling(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    n0 = launch_count()
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        for _ in range(args.steps):
            tr.step_async(sc)
        ev1.record()
        torch.cuda.synchronize()
    tr.sync()
    launches = launch_count() - n0
    ms = ev0.elapsed_time(ev1)
    phase_ms, n_prof = tr.get_timings()
    tr.set_profiling(False)
    if args.dump_outputs:  # before the e2e leg below trains the same factors further
        dump_outputs(args.dump_outputs, tr.user, tr.item)
    value = w["nnz"] * args.steps / (ms / 1e3)

    # ---- end to end through the reference-facing API, host buffers ----
    pin = [torch.empty((w["n_users"], w["K"]), dtype=torch.float32, pin_memory=True),
           torch.empty((w["n_items"], w["K"]), dtype=torch.float32, pin_memory=True)]
    host = [p.numpy() for p in pin]
    host[0][:] = tr.user
    host[1][:] = tr.item
    e2e_steps = max(3, min(args.steps, 10))

    def e2e_step():
        # H2D of both factor matrices from pinned host memory, IALSTrainer.step (synchronous,
        # checks the solver status), D2H of both into the same pinned buffers: one C-ABI call
        # (ials_trainer_step_io) so that the user read-back overlaps the item half-epoch
        tr.step_io(sc, host[0], host[1])

    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_dt = time.perf_counter() - t0
    factor_bytes = (w["n_users"] + w["n_items"]) * w["K"] * 4

    # ---- roofline of the dominant kernel ----
    # cg_rows_kernel (one launch per half-epoch) solves every row that is not "heavy";
    # its algorithmic bytes: each neighbour's K-vector + int32 index + f32 value once, the
    # row's own vector read + written, indptr (DESIGN.md "Algorithmic bytes").
    peak, peak_kind = measured_peaks()
    n_ep = max(n_prof, 1)
    ph = [v / n_ep for v in phase_ms]
    names = ["gram_item", "users_heavy_wgram", "users_heavy_dense_cg", "users_light_cg",
             "gram_user", "items_heavy_wgram", "items_heavy_dense_cg", "items_light_cg"]
    plan = [tr.plan_stats(0), tr.plan_stats(1)]
    K = w["K"]
    light_bytes = 0
    for p in plan:
        light_bytes += ((p["nnz"] - p["heavy_nnz"]) * (4 * K + 8)
                        + (p["rows"] - p["heavy_rows"]) * 8 * K + (p["rows"] + 1) * 8)
    light_ms = ph[3] + ph[7]
    achieved = light_bytes / (light_ms / 1e3) / 1e9
    solve_ms = sum(ph[1:4]) + sum(ph[5:8])
    light_kernel = "cg_rows_kernel"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")  # from the committed ncu --set full capture
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(f"{light_kernel}_dram_bytes_per_launch")
    roofline = {
        "bound": "hbm", "kernel": f"{light_kernel} (2 launches per epoch: users, items)",
        "achieved": achieved, "peak": peak, "peak_kind": peak_kind, "unit": "GB/s",
        "frac": achieved / peak, "traffic": traffic,
        "algorithmic_bytes_per_launch": light_bytes / 2, "ms_per_launch": light_ms / 2,
        "share_of_step": light_ms / (ms / args.steps),
        "phases_ms_per_epoch": dict(zip(names, ph)),
        "schedule": {"users": plan[0], "items": plan[1]},
        "whole_solve": {"algorithmic_bytes_per_epoch": solve_bytes(w), "ms_per_epoch": solve_ms,
                        "achieved": solve_bytes(w) / (solve_ms / 1e3) / 1e9,
                        "frac": solve_bytes(w) / (solve_ms / 1e3) / 1e9 / peak},
        "epoch_algorithmic_gbs": epoch_bytes(w) / (ms / args.steps / 1e3) / 1e9,
    }

    # ---- configs[3] on this one GPU: the strong-scaling reference of the N > 1 lines ----
    c4 = None
    if args.c4 != "off":
        del tr
        torch.cuda.empty_cache()
        try:
            from irspack_b200 import dist as ials_dist

            c4 = ials_dist.run_c4(HYPER, steps=2, warmup=1, scale=float(os.environ.get("IALS_BENCH_C4_SCALE", "1.0")),
                                  e2e_steps=1, score_users_per_rank=65536, parity_check=oracle_row_check)
            c4["what"] = ("BASELINE configs[3] (and the configs[4] top-100 sample) on ONE B200: the whole "
                          "1 B-interaction matrix, same code path as bench.py --gpus N")
        except Exception as e:  # the headline line must survive a failure of the side run
            c4 = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- CPU baseline: the oracle port on this box's cores, whole workload ----
    import oracle

    nt = oracle.hardware_threads()
    cpu_t = cpu_epochs(w, X, u0, i0, args.cpu_epochs, nt)
    cpu_value = w["nnz"] / float(np.median(cpu_t))

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "epochs_per_sec": args.steps / (ms / 1e3),
        "config": config_dict(w, 1),
        "clocks": clocks.summary(),
        "e2e": {"value": w["nnz"] * e2e_steps / e2e_dt, "unit": UNIT,
                "h2d_bytes_per_step": factor_bytes, "d2h_bytes_per_step": factor_bytes,
                "ms_per_step": 1e3 * e2e_dt / e2e_steps, "steps": e2e_steps,
                "what": "IALSTrainer.step_io: upload user+item from pinned host, one epoch, read both back "
                        "(the user warm starts arrive in 2 MB chunks, flagged by the copy engine, while the "
                        "user half-epoch takes its rows in arrival order; user read-back overlapped with the "
                        "item half-epoch)"},
        "gpu_launches": int(launches),
        "roofline": roofline,
        "cpu_baseline": {"value": cpu_value, "unit": UNIT, "cores": nt, "kind": "port",
                         "sample": f"median of {args.cpu_epochs} full epochs of the same matrix "
                                   f"and initial factors (after 1 warm-up epoch)",
                         "ms_per_epoch": 1e3 * float(np.median(cpu_t))},
        "c4_single_gpu": c4,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--cpu-epochs", type=int, default=5)
    ap.add_argument("--c4", choices=["auto", "off"], default="auto",
                    help="N=1 only: also time configs[3] (1 B interactions) on the one GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="--gpus 1 only: write the factors of the last timed epoch to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus != 1:
        ap.error("--dump-outputs is implemented for --gpus 1")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
