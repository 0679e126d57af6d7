#!/usr/bin/env python
"""Times explanations (``ials_trainer_explain``).

    python tools/time_explain.py [--reps 5] [--out profiles/r03f_explain.json]

(a) The configs[1] shape (138 493 x 26 744, 20 M interactions from ``synth_csr``, K = 128): 32 768 users
    by index, each explaining its own top-10 of ``recommend_users`` (training items masked), n_top = 10.
(b) The same on the configs[2] shape (480 189 x 17 770, 100 M interactions) at K = 256.
(c) On each model, the 64 heaviest users alone: the per-CTA worst case (one CTA solves one user).

Each timed call is warmed up first and ends in a device synchronise (host checks, uploads, the Gram of
the item side, the kernels and the copies back).  Reported: median / min call time, the algorithmic FLOPs
sum_u (nnz_u K^2 / 2 + K^3 / 3 + 2 T K^2 + T nnz_u K) and their rate, and from a separate run under
``torch.profiler`` the device time per kernel (the Gram, the explain kernel, the top-k).  The card's
name, power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from time_candidates import card, kernel_split, timed  # noqa: E402

N_QUERY, T, N_TOP = 32_768, 10, 10


def flops(nnz: np.ndarray, K: int, t: int) -> float:
    nnz = nnz.astype(np.float64)
    return float(np.sum(nnz * K * K / 2 + K ** 3 / 3 + 2 * t * K * K + t * nnz * K))


def workload(core, shape: str, seed: int, reps: int) -> dict:
    from irspack_b200.synth import SHAPES, init_factors, synth_csr

    U, I, nnz, K = SHAPES[shape]
    X = synth_csr(U, I, nnz, seed)
    cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.02).build()
    tr = core.IALSTrainer(cfg, X)
    tr.user, tr.item = init_factors(U, K, seed + 1), init_factors(I, K, seed + 2)
    deg = np.diff(X.indptr)
    rng = np.random.default_rng(seed + 3)
    out = {"shape": shape, "users": U, "items": I, "nnz": nnz, "K": K, "n_top": N_TOP, "targets_per_user": T}
    cases = {"a_32768_users": rng.choice(U, N_QUERY, replace=False).astype(np.int64),
             "c_64_heaviest": np.argsort(-deg, kind="stable")[:64].astype(np.int64)}
    for name, q in cases.items():
        top, cnt = tr.recommend_users(q, T, mask="train")
        targets = [top[r, :cnt[r]] for r in range(q.size)]
        call = lambda: tr.explain(0, q, targets, n_top=N_TOP)  # noqa: E731
        call()
        ts = [timed(call) for _ in range(reps)]
        f = flops(deg[q], K, T)
        med = float(np.median(ts))
        out[name] = {"queries": int(q.size), "history_nnz": int(deg[q].sum()), "max_history": int(deg[q].max()),
                     "median_s": med, "min_s": float(np.min(ts)), "algorithmic_flop": f,
                     "algorithmic_tflops_at_median": f / med / 1e12,
                     "kernels_ms_profiled": kernel_split(call)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03f_explain.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("time_explain.py needs a CUDA device")
    from irspack_b200 import _ials_core as core

    res = {"card": card()}
    res["configs1_K128"] = workload(core, "ml20m", 1, args.reps)
    print(json.dumps(res, indent=1), flush=True)
    res["configs2_K256"] = workload(core, "netflix", 2, args.reps)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
