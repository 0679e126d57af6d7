#!/usr/bin/env python
"""Evaluation passes of the row-sharded trainer.  Prints one JSON line (rank 0).

configs[3] shape (the 1 B-interaction power-law matrix, 10 M x 2 M, K = 128) row-sharded over the
ranks of the process group (``torchrun --nproc-per-node N``; one GPU without it), with a held-out set
of 10 items per user drawn on the device from a seed of its own: one ``ShardedEvaluator`` pass (nDCG
and the other metrics at 10 and 100 over every user of every rank) against a lists-only pass over the
same users (the ``recommend`` loop of ``run_c4``, top-100 with the training mask), the pass split into
list production, metrics kernels, all-reduce and diversity kernels (device times from a profiled pass
of their own), and one save_state / load_state.  The factors are the random initial ones: the pass
costs the same for any factors.

configs[1] (ML-20M shape) on one GPU, in the same call: the world-1 ShardedEvaluator pass against
``Evaluator.get_score`` on an ``IALSRecommender`` with the same factors; the two dicts must agree to
1e-12.

    python tools/time_sharded_eval.py [--scale 1.0] [--repeats 3] [--out profiles/x.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GROUPS = {  # device-kernel name fragments of each part of a pass
    "lists": ("score_tc_kernel", "merge_topk_kernel", "score_tile_kernel", "topk_rows_kernel", "mask_rows_kernel"),
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
    out["other"] = 0.0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3
        if t <= 0:
            continue
        group = next((g for g, names in GROUPS.items() if any(n in e.key for n in names)), "other")
        out[group] += t
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--gt-per-user", type=int, default=10)
    ap.add_argument("--block", type=int, default=262144, help="users per recommend call of the lists-only loop")
    ap.add_argument("--skip-c1", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()

    import numpy as np
    import torch
    import torch.distributed as dist

    from bench import HYPER
    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import (ShardedEvaluator, ShardedIALSTrainer, c4_shape, exchange_transposed_shards_device,
                                   global_item_bounds_device, synth_user_block_device)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    rank = dist.get_rank() if world > 1 else 0
    dev = torch.device(f"cuda:{local}")

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier() -> None:
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                          "-i", str(local)], capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu, "world": world}

    # ---- configs[3] shape, row-sharded ----
    U, I, nnz, K = c4_shape(a.scale, world)
    ub = np.linspace(0, U, world + 1).astype(np.int64)
    nb = np.linspace(0, nnz, world + 1).astype(np.int64)
    n_rows, n_nnz = int(ub[rank + 1] - ub[rank]), int(nb[rank + 1] - nb[rank])
    ip, ix, dt = synth_user_block_device(n_rows, I, n_nnz, seed=1004 + rank, device=dev, item_seed=1004)
    bounds = global_item_bounds_device(ix, I)
    t_csr = exchange_transposed_shards_device(ip, ix, dt, int(ub[rank]), U, bounds)
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(HYPER["alpha0"]).set_reg(HYPER["reg"])
           .set_nu(HYPER["nu"]).build())
    tr = ShardedIALSTrainer(cfg, (ip, ix, dt), int(ub[rank]), U, t_csr, int(bounds[rank]), I, init_on_device=True)
    del ip, ix, dt, t_csr
    # held-out: 10 items per user from a seed of its own (the same popularity law)
    gt = synth_user_block_device(n_rows, I, n_rows * a.gt_per_user, seed=77_000 + rank, device=dev, item_seed=1004)
    torch.cuda.empty_cache()
    sev = ShardedEvaluator(tr, gt)
    del gt
    cutoffs = [10, 100]
    b0, b1 = tr.user_range
    idx = np.empty((a.block, 100), dtype=np.int32)
    cnt = np.empty((a.block,), dtype=np.int32)

    def lists_only() -> None:
        for b in range(b0, b1, a.block):
            m = min(a.block, b1 - b)
            tr.recommend(b, b + m, 100, idx[:m], cnt[:m])

    def evaluate():
        return sev.get_scores(tr, cutoffs)

    lists_only()
    scores = evaluate()  # warm-up: scratch, the set, the diversity workspace
    runs = []
    for _ in range(a.repeats):
        barrier()
        t0 = time.perf_counter()
        lists_only()
        torch.cuda.synchronize()
        t_lists = max_over_ranks(time.perf_counter() - t0)
        barrier()
        t0 = time.perf_counter()
        again = evaluate()
        t_eval = max_over_ranks(time.perf_counter() - t0)
        assert again == scores, "two passes over the same model differ"
        split = {k: max_over_ranks(v) for k, v in sev.last_timings.items()}
        runs.append({"lists_only_s": t_lists, "evaluate_s": t_eval, "host_split_s": split})
    dev_ms = kernel_ms(evaluate, torch)
    dev_ms = {k: max_over_ranks(v) for k, v in dev_ms.items()}
    # save_state / load_state of the rank's own rows (pinned host buffers)
    state = tr.save_state()
    barrier()
    t0 = time.perf_counter()
    state = tr.save_state(state)
    t_save = max_over_ranks(time.perf_counter() - t0)
    barrier()
    t0 = time.perf_counter()
    tr.load_state(state)
    t_load = max_over_ranks(time.perf_counter() - t0)
    best = min(runs, key=lambda r: r["evaluate_s"])
    res["configs3"] = {
        "n_users": U, "n_items": I, "nnz": nnz, "K": K, "held_out_per_user": a.gt_per_user, "cutoffs": cutoffs,
        "users_per_s": U / best["evaluate_s"], "best": best, "runs": runs,
        "device_ms_one_pass_max_over_ranks": dev_ms,
        "metrics_merge_diversity_over_lists_only": (best["evaluate_s"] - best["lists_only_s"]) / best["lists_only_s"],
        "save_state_s": t_save, "load_state_s": t_load,
        "scores": {k: v for k, v in scores.items() if k.split("@")[0] in ("ndcg", "recall", "hit", "appeared_item")},
        "what": "seconds are host wall clock around the call, max over ranks; lists_only = ials_trainer_recommend "
                "(k = 100, training mask) in blocks incl. the D2H of the lists; evaluate = "
                "ShardedEvaluator.get_scores([10, 100]); device_ms from a separate profiled pass",
    }
    del sev, tr
    torch.cuda.empty_cache()

    # ---- configs[1] on one GPU: world-1 ShardedEvaluator against Evaluator(IALSRecommender) ----
    if world == 1 and not a.skip_c1:
        from irspack_b200 import Evaluator, IALSRecommender
        from irspack_b200.synth import SHAPES, holdout_split, synth_csr

        U1, I1, nnz1, K1 = SHAPES["ml20m"]
        X = synth_csr(U1, I1, nnz1, seed=3)
        X_tr, X_te = holdout_split(X, 0.2, seed=4)
        rec = IALSRecommender(X_tr, n_components=K1, alpha0=HYPER["alpha0"], reg=HYPER["reg"],
                              train_epochs=4).learn()
        cfg1 = core.IALSModelConfigBuilder().set_K(K1).build()
        tr1 = ShardedIALSTrainer.from_global(cfg1, X_tr, rank=0, world=1)
        tr1.user, tr1.item = rec.get_user_embedding(), rec.get_item_embedding()
        ev, sev1 = Evaluator(X_te), ShardedEvaluator.from_global(tr1, X_te)
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
        res["configs1"] = {"n_users": U1, "n_items": I1, "cutoff": 10, "evaluator_ms": 1e3 * min(t_ev),
                           "sharded_evaluator_ms": 1e3 * min(t_sev), "max_rel_diff": rel,
                           "equal_to_1e-12": bool(rel <= 1e-12), "ndcg@10": got["ndcg"]}
    if rank == 0:
        line = json.dumps(res)
        print(line, flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(line + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
