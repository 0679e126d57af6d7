#!/usr/bin/env python
"""Times candidate ranking (``ials_trainer_rank_candidates``).

    python tools/time_candidates.py [--reps 5] [--out profiles/r03e_candidates.json]

(a) The configs[1] catalogue (26 744 items, K = 128; L2-resident), 32 768 users picked by index with
    100 candidates each, top-10 without a mask (factors-only trainer).  Timed alternately with
    ``recommend_users`` given the same lists as allow-lists (the fused tensor-core route, which scores
    the whole catalogue), and both routes' lists are compared (equal, or swapped within float32 ties).
    The same with 256 and 257 candidates each: the two sides of the list length at which the selection
    changes from a warp per list (<= 256) to a CTA per list.
(b) A 2 M-item, K = 128 catalogue (larger than L2), the users [0, 1 M) with 1 000 candidates each
    (one random item in each block of 2 000 ids), at k = 100 and k = 1 000, through the C ABI (the
    lists are generated strictly ascending, so the Python layer's sorting has nothing to do).

Each timed call is warmed up first and ends in a device synchronise (the lists are copied to the host
inside the call; the call time includes the host-side list checks and the upload of the candidates).
Reported: median / min call time, pairs/s, and the gathered item-row bytes (pairs x 512 B) per second
against the data-sheet 7.7 TB/s.  A separate run under ``torch.profiler`` gives the device time of the
two kernels.  The card's name, power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

HBM_TBPS = 7.7
K = 128


def card(device: int = 0) -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def model(core, n_users: int, n_items: int, seed: int):
    rng = np.random.default_rng(seed)
    cfg = core.IALSModelConfigBuilder().set_K(K).build()
    return core.IALSTrainer._from_factors(cfg, 0.1 * rng.standard_normal((n_users, K), dtype=np.float32),
                                          0.1 * rng.standard_normal((n_items, K), dtype=np.float32))


def timed(fn) -> float:
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def stats(ts, pairs: int) -> dict:
    med = float(np.median(ts))
    return {"median_s": med, "min_s": float(np.min(ts)), "pairs_per_s": pairs / med,
            "gathered_bytes_per_s": pairs * K * 4 / med, "of_hbm_datasheet": pairs * K * 4 / med / (HBM_TBPS * 1e12)}


def kernel_split(fn) -> dict:
    """Device time per kernel name (ms) of one call of fn under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t and ("kernel" in e.key or "Memcpy" in e.key):
            out[e.key[:80]] = out.get(e.key[:80], 0.0) + t / 1e3
    return out


def rank_c_abi(core, tr, begin, end, k, ip, ix):
    rows = end - begin
    idx = np.empty((rows, k), np.int32)
    sc = np.empty((rows, k), np.float32)
    cnt = np.empty(rows, np.int32)
    p = core._ptr
    core.check(core.lib.ials_trainer_rank_candidates(tr._handle, None, None, begin, end, k, 1, None, None, rows,
                                                     p(ip), p(ix), p(idx), p(sc), p(cnt)))
    return idx, cnt, sc


def workload_a(core, tr, reps: int, n_c: int) -> dict:
    U, I, n_q, k = 138_493, 26_744, 32_768, 10
    rng = np.random.default_rng(2)
    q = rng.integers(0, U, size=n_q).astype(np.int64)
    ix = np.concatenate([np.sort(rng.choice(I, n_c, replace=False)) for _ in range(n_q)]).astype(np.int32)
    ip = np.arange(n_q + 1, dtype=np.int64) * n_c
    lists = (n_q, ip, ix)
    rank = lambda: tr.rank_candidates(q, lists, k, mask=None)  # noqa: E731
    fused = lambda: tr.recommend_users(q, k, mask=None, return_scores=True, allowed=lists)  # noqa: E731
    for f in (rank, fused):
        f()
    t_rank, t_fused = [], []
    for _ in range(reps):
        t_rank.append(timed(rank))
        t_fused.append(timed(fused))
    (idx, cnt, sc), (fidx, fcnt, fsc) = rank(), fused()
    same_rows = int(np.sum(np.all(idx == fidx, axis=1)))
    max_score_diff = float(np.abs(sc - fsc).max())
    pairs = n_q * n_c
    return {"users": n_q, "items": I, "K": K, "candidates_per_user": n_c, "k": k, "pairs": pairs,
            "rank_candidates": stats(t_rank, pairs), "recommend_users_allowed_fused": stats(t_fused, pairs),
            "fused_over_candidates": float(np.median(t_fused) / np.median(t_rank)),
            "lists_identical_rows": same_rows, "counts_equal": bool(np.array_equal(cnt, fcnt)),
            "max_abs_score_diff": max_score_diff,
            "kernels_ms_profiled_rank": kernel_split(rank), "kernels_ms_profiled_fused": kernel_split(fused)}


def workload_b(core, reps: int) -> dict:
    U, I, n_c = 1_000_000, 2_000_000, 1000
    tr = model(core, U, I, 3)
    rng = np.random.default_rng(4)
    block = I // n_c
    ix = rng.integers(0, block, size=(U, n_c), dtype=np.int32)
    ix += (np.arange(n_c, dtype=np.int32) * block)[None, :]
    ix = ix.reshape(-1)
    ip = np.arange(U + 1, dtype=np.int64) * n_c
    pairs = U * n_c
    out = {"users": U, "items": I, "K": K, "candidates_per_user": n_c, "pairs": pairs, "cutoffs": {}}
    for k in (100, 1000):
        call = lambda: rank_c_abi(core, tr, 0, U, k, ip, ix)  # noqa: E731
        call()
        ts = [timed(call) for _ in range(reps)]
        out["cutoffs"][str(k)] = {**stats(ts, pairs), "kernels_ms_profiled": kernel_split(call)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03e_candidates.json"))
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("time_candidates.py needs a CUDA device")
    from irspack_b200 import _ials_core as core

    tr = model(core, 138_493, 26_744, 1)
    res = {"card": card(), "hbm_datasheet_tbps": HBM_TBPS,
           "a_configs1_catalogue": {str(n_c): workload_a(core, tr, args.reps, n_c) for n_c in (100, 256, 257)}}
    print(json.dumps(res["a_configs1_catalogue"], indent=1), flush=True)
    del tr
    res["b_2m_catalogue"] = workload_b(core, max(2, args.reps // 2))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
