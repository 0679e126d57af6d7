#!/usr/bin/env python
"""Cold-user evaluation passes of the row-sharded trainer at world 1.  Prints one JSON line.

configs[1] (ML-20M shape): 10 % of the users are held out of training; 80 % of each held-out row is
the fold-in input and 20 % the ground truth.  One ``ShardedEvaluatorWithColdUser`` pass (nDCG@10 and
the rest) against ``EvaluatorWithColdUser.get_score`` on an ``IALSRecommender`` with the same factors
and model configuration; the two dicts must agree to 1e-12.

configs[3]-shaped model (10 M users x 2 M items, K = 128, random item factors) and 1 M cold users with
100 interactions each (the configs[3] mean) and 10 held-out items each, from the power-law generator:
one pass at cutoffs 10 and 100, its wall time and its device time split into fold-in (Gram of the item
factors and the row solves), list production, metrics and diversity kernels (a profiled pass of its
own).  The cold pass reads the item factors and the cold users only, so the model is built without a
training matrix.

    python tools/time_sharded_cold_eval.py [--repeats 3] [--cold-users 1000000] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GROUPS = {  # device-kernel name fragments of each part of a pass; the rest is the fold-in
    "lists": ("score_tc_kernel", "merge_topk_kernel", "score_tile_kernel", "topk_rows_kernel", "mask_rows_kernel",
              "allow_rows_kernel"),
    "metrics": ("metrics_rows_kernel", "metrics_reduce_kernel"),
    "diversity": ("hist_stats_kernel", "count_of_counts_kernel", "table_block_sums_kernel", "table_terms_kernel",
                  "diversity_finish_kernel"),
}


def kernel_ms(fn, torch):
    """Device milliseconds per group of one call of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in GROUPS}
    out["fold_in"] = 0.0
    names = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
        if t <= 0:
            continue
        group = next((g for g, frags in GROUPS.items() if any(n in e.key for n in frags)), "fold_in")
        out[group] += t
        if group == "fold_in":
            names[e.key[:80]] = round(t, 3)
    out["fold_in_parts"] = names
    return out


def cold_split(X, fraction, input_share, seed):
    """(warm rows, cold input, cold ground truth): `fraction` of the users drawn at random are cold, and
    `input_share` of each cold row's entries (drawn at random) is its input, the rest its ground truth."""
    import numpy as np
    import scipy.sparse as sps

    rng = np.random.default_rng(seed)
    U = X.shape[0]
    cold = np.zeros(U, dtype=bool)
    cold[rng.choice(U, int(round(fraction * U)), replace=False)] = True
    C = sps.csr_matrix(X[cold])
    keep = rng.random(C.nnz) < input_share
    rows = np.repeat(np.arange(C.shape[0]), np.diff(C.indptr))

    def part(m):
        return sps.csr_matrix((C.data[m], (rows[m], C.indices[m])), shape=C.shape)

    return sps.csr_matrix(X[~cold]), part(keep), part(~keep)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cold-users", type=int, default=1_000_000)
    ap.add_argument("--per-user", type=int, default=100)
    ap.add_argument("--gt-per-user", type=int, default=10)
    ap.add_argument("--skip-c1", action="store_true")
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import scipy.sparse as sps
    import torch

    from bench import HYPER
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import ShardedEvaluatorWithColdUser, ShardedIALSTrainer, synth_user_block_device

    torch.cuda.set_device(0)
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", "0"], capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "world": 1}
    # the prediction-time solver of ials.IALSTrainer (CG, 5 steps)
    sc = core.IALSSolverConfigBuilder().set_max_cg_steps(5).set_ialspp_iteration(7).build()

    # ---- configs[1]: world-1 ShardedEvaluatorWithColdUser against EvaluatorWithColdUser(IALSRecommender) ----
    if not a.skip_c1:
        from irspack_b200 import EvaluatorWithColdUser, IALSRecommender
        from irspack_b200.synth import SHAPES, synth_csr

        U1, I1, nnz1, K1 = SHAPES["ml20m"]
        X = synth_csr(U1, I1, nnz1, seed=3)
        X_warm, X_in, X_gt = cold_split(X, 0.1, 0.8, seed=4)
        rec = IALSRecommender(X_warm, n_components=K1, alpha0=HYPER["alpha0"], reg=HYPER["reg"], nu=HYPER["nu"],
                              train_epochs=4).learn()
        cfg1 = (core.IALSModelConfigBuilder().set_K(K1).set_alpha0(HYPER["alpha0"]).set_reg(HYPER["reg"])
                .set_nu(HYPER["nu"]).build())
        tr1 = ShardedIALSTrainer.from_global(cfg1, X_warm, rank=0, world=1)
        tr1.user, tr1.item = rec.get_user_embedding(), rec.get_item_embedding()
        ev = EvaluatorWithColdUser(X_in, X_gt)
        sev1 = ShardedEvaluatorWithColdUser(tr1, X_in, X_gt, sc)
        want, got = ev.get_score(rec), sev1.get_score(tr1)
        t_ev, t_sev = [], []
        for _ in range(a.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ev.get_score(rec)
            t_ev.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            sev1.get_score(tr1)
            t_sev.append(time.perf_counter() - t0)
        rel = max(abs(got[k] - want[k]) / max(abs(want[k]), 1e-300) for k in want)
        res["configs1"] = {
            "n_users_warm": X_warm.shape[0], "n_cold_users": X_in.shape[0], "n_items": I1, "K": K1,
            "input_nnz": int(X_in.nnz), "ground_truth_nnz": int(X_gt.nnz), "cutoff": 10,
            "evaluator_with_cold_user_ms": 1e3 * min(t_ev), "sharded_cold_evaluator_ms": 1e3 * min(t_sev),
            "max_rel_diff": rel, "equal_to_1e-12": bool(rel <= 1e-12), "ndcg@10": got["ndcg"],
            "what": "host wall clock of get_score, best of the repeats, after a warm-up call",
        }
        del sev1, tr1, rec
        torch.cuda.empty_cache()

    # ---- configs[3]-shaped model, 1 M cold users ----
    if not a.skip_c3:
        U, I, _, K = (10_000_000, 2_000_000, 0, 128)
        cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(HYPER["alpha0"]).set_reg(HYPER["reg"])
               .set_nu(HYPER["nu"]).build())
        tr = ShardedIALSTrainer(cfg, sps.csr_matrix((U, I), dtype=np.float32), 0, U,
                                sps.csr_matrix((I, U), dtype=np.float32), 0, I, init_on_device=True)
        C = a.cold_users

        def host_csr(triple, n):
            ip, ix, dt = (t.cpu().numpy() for t in triple)
            return sps.csr_matrix((dt, ix, ip), shape=(n, I))

        X_in = host_csr(synth_user_block_device(C, I, C * a.per_user, seed=5004, device=dev, item_seed=1004), C)
        X_gt = host_csr(synth_user_block_device(C, I, C * a.gt_per_user, seed=77_004, device=dev,
                                                item_seed=1004), C)
        torch.cuda.empty_cache()
        t0 = time.perf_counter()
        sev = ShardedEvaluatorWithColdUser(tr, X_in, X_gt, sc)
        t_build = time.perf_counter() - t0
        cutoffs = [10, 100]

        def evaluate():
            return sev.get_scores(tr, cutoffs)

        t0 = time.perf_counter()
        scores = evaluate()  # warm-up: the set (upload, validation, plan), scratch, the diversity workspace
        t_first = time.perf_counter() - t0
        runs = []
        for _ in range(a.repeats):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            again = evaluate()
            runs.append(time.perf_counter() - t0)
            assert again == scores, "two passes over the same model differ"
        dev_ms = kernel_ms(evaluate, torch)
        best = min(runs)
        res["configs3"] = {
            "n_users_model": U, "n_items": I, "K": K, "n_cold_users": C, "input_nnz": int(X_in.nnz),
            "ground_truth_nnz": int(X_gt.nnz), "cutoffs": cutoffs, "pass_s": best, "runs_s": runs,
            "cold_users_per_s": C / best, "first_call_s": t_first, "evaluator_build_s": t_build,
            "device_ms_one_pass": dev_ms, "host_split_s": sev.last_timings,
            "scores": {k: v for k, v in scores.items() if k.split("@")[0] in ("ndcg", "recall", "hit", "appeared_item")},
            "what": "pass_s: host wall clock of ShardedEvaluatorWithColdUser.get_scores([10, 100]) at world 1, best "
                    "of the repeats after the first call (which builds the evaluation set); device_ms from a "
                    "separate profiled pass; the model's training matrix is empty: the pass reads only the item "
                    "factors (random) and the cold users",
        }
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
