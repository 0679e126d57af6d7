#!/usr/bin/env python
"""Per-epoch milliseconds of feature-aware iALS on the BASELINE configs[1] shape (ML-20M:
138 493 x 26 744, 20 M interactions, K = 128, CG, max_cg_steps = 3) with 300 dense item features
and sparse user features: the single-GPU IALSTrainer against the row-sharded trainer on one rank
(world 1), each with and without features, plus the device time of the sharded trainer's weight
refits (ShardedIALSTrainer._refit: partial sums, their all-reduce -- none at world 1 -- and the
ridge solve).  Prints one JSON line.

    python tools/time_sharded_features.py [--steps 5] [--warmup 2] [--scale 1.0]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--user-features", type=int, default=64)
    ap.add_argument("--user-feature-nnz", type=int, default=5, help="stored entries per user feature row")
    ap.add_argument("--item-features", type=int, default=300)
    a = ap.parse_args()

    import numpy as np
    import scipy.sparse as sps
    import torch

    from bench import HYPER
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedIALSTrainer
    from irspack_b200.synth import SHAPES, init_factors, synth_csr

    U, I, nnz, K = SHAPES["ml20m"]
    U, nnz = int(U * a.scale), int(nnz * a.scale)
    X = synth_csr(U, I, nnz, seed=1002)
    rng = np.random.default_rng(0)
    cols = rng.integers(0, a.user_features, (U, a.user_feature_nnz))
    uf = sps.csr_matrix((rng.standard_normal(cols.size).astype(np.float32),
                         (np.repeat(np.arange(U), a.user_feature_nnz), cols.ravel())), shape=(U, a.user_features))
    uf.sum_duplicates()
    itf = rng.standard_normal((I, a.item_features)).astype(np.float32)
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(HYPER["alpha0"]).set_reg(HYPER["reg"])
           .set_nu(HYPER["nu"]).set_lambda_user_feature(1.0).set_lambda_item_feature(1.0).build())
    sc = core.IALSSolverConfigBuilder().set_max_cg_steps(HYPER["max_cg_steps"]).build()
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    feats = {"user_feature": uf, "item_feature": itf}

    def make(kind: str, with_features: bool):
        if kind == "single":
            t = core.IALSTrainer(cfg, X, uf, itf) if with_features else core.IALSTrainer(cfg, X)
        else:
            t = ShardedIALSTrainer.from_global(cfg, X, rank=0, world=1, **(feats if with_features else {}))
        t.user, t.item = u0, i0
        return t

    def time_epochs(t):
        for _ in range(a.warmup):
            t.step(sc)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record()
        for _ in range(a.steps):
            t.step_async(sc)
        ev1.record()
        t.sync()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3 / a.steps
        return ev0.elapsed_time(ev1) / a.steps, wall

    res = {}
    for kind in ("single", "sharded_world1"):
        for with_features in (False, True):
            t = make(kind, with_features)
            refit = []
            if kind != "single" and with_features:  # device time of every refit of the timed epochs
                inner = t._refit

                def timed_refit(side, inner=inner, refit=refit):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    inner(side)
                    e1.record()
                    refit.append((side, e0, e1))

                t._refit = timed_refit
            ms, wall = time_epochs(t)
            key = f"{kind}_{'features' if with_features else 'plain'}"
            res[key] = {"ms_per_epoch_events": round(ms, 3), "ms_per_epoch_wall": round(wall, 3)}
            if refit:
                timed = refit[-2 * a.steps:]
                per_side = [sum(e0.elapsed_time(e1) for s, e0, e1 in timed if s == side) / a.steps for side in (0, 1)]
                res[key]["refit_ms_per_epoch"] = {"user": round(per_side[0], 3), "item": round(per_side[1], 3)}
            res[key]["loss"] = t.compute_loss(sc)
            del t
            torch.cuda.empty_cache()
    ld = 128
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    print(json.dumps({
        "shape": {"users": U, "items": I, "nnz": int(X.nnz), "K": K, "solver": "CG", "max_cg_steps": 3},
        "features": {"user": f"CSR {a.user_features} columns, ~{a.user_feature_nnz} entries per row",
                     "item": f"dense {a.item_features} columns"},
        "steps": a.steps, "warmup": a.warmup, "gpu": gpu, "results": res,
        "refit_allreduce_bytes_per_epoch": {"user": a.user_features * ld * 4, "item": a.item_features * ld * 4},
        "refit_allreduce_bytes_first_epoch_extra": {"user": a.user_features ** 2 * 4,
                                                    "item": a.item_features ** 2 * 4},
        "note": "world 1 runs no collective: the all-reduce time of the refit buffers on several GPUs is not "
                "measured here",
    }), flush=True)


if __name__ == "__main__":
    main()
