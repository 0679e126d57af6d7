#!/usr/bin/env python
"""Times similar-item lists (``IALSTrainer.similar``, ``ials_trainer_similar``).

    python tools/time_similar.py [--reps 3] [--gpus N] [--out profiles/r03d_similar.json]

1. The whole neighbour graph of a 2 M-item catalogue at K = 128 (synthetic factors from a seed): the
   top-100 cosine neighbours of every item.  Alternating with it, a ``recommend`` pass of 2 M user
   rows against the same catalogue (no mask, top-100): the same product and top-k, so the difference
   between the two is what the similarity pass adds (the unit-norm copy and the self mask).  One more
   similarity pass runs under ``torch.profiler`` for the device time of each kernel.
2. Every item of the configs[1] catalogue (26 744 items, K = 128), top-10.
3. The same at K = 256 (the fused kernel's WIDE layout).
4. With ``--gpus N`` (N > 1): the 2 M-item graph split over N GPUs, each taking its
   ``balanced_bounds`` range of items on a full copy of the factors; the pass time is the slowest
   rank's.  Not run on one GPU.

Each timed pass is warmed up first and ends in a device synchronise (the lists are copied to the
host inside the call).  Times are the median and minimum of ``--reps`` passes; the algorithmic rate is
2 n_queries n_catalogue K / t.  The card's name, power limit and max SM clock are read in the same run.
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

BIG_ITEMS, BIG_K, BIG_CUTOFF = 2_000_000, 128, 100
C1_ITEMS, C1_CUTOFF = 26_744, 10


def card(device: int = 0) -> dict:
    q = subprocess.run(["nvidia-smi", f"--id={device}", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def factors(n: int, K: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return (0.1 * rng.standard_normal((n, K), dtype=np.float32)).astype(np.float32)


def model(core, n_users: int, n_items: int, K: int, seed: int):
    cfg = core.IALSModelConfigBuilder().set_K(K).build()
    return core.IALSTrainer._from_factors(cfg, factors(n_users, K, seed), factors(n_items, K, seed + 1))


def timed(fn) -> float:
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def stats(seconds, flop: float) -> dict:
    med = float(np.median(seconds))
    return {"median_s": med, "min_s": float(np.min(seconds)), "s": [round(x, 4) for x in seconds],
            "tflops_algorithmic": flop / med / 1e12}


def kernel_profile(fn) -> dict:
    """Device time per kernel name (ms) of one call of fn, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key[:80]] = round(t / 1e3, 3)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def big_graph(core, reps: int) -> dict:
    tr = model(core, BIG_ITEMS, BIG_ITEMS, BIG_K, seed=11)
    flop = 2.0 * BIG_ITEMS * BIG_ITEMS * BIG_K
    sim = lambda: tr.similar(1, None, BIG_CUTOFF)  # noqa: E731
    rec = lambda: tr.recommend(0, BIG_ITEMS, BIG_CUTOFF, mask=None, return_scores=True)  # noqa: E731
    sim()
    rec()
    ts, tr_ = [], []
    for _ in range(reps):  # alternating
        ts.append(timed(sim))
        tr_.append(timed(rec))
    idx, cnt, sc = tr.similar(1, None, BIG_CUTOFF)
    out = {"items": BIG_ITEMS, "K": BIG_K, "cutoff": BIG_CUTOFF, "metric": "cosine",
           "similar_all_items": stats(ts, flop), "recommend_2M_user_rows": stats(tr_, flop),
           "similar_over_recommend": float(np.median(ts) / np.median(tr_)),
           "counts_all_full": bool(np.all(cnt == BIG_CUTOFF)), "self_in_lists": int((idx == np.arange(BIG_ITEMS)[:, None]).sum())}
    del idx, cnt, sc
    out["similar_kernel_ms"] = kernel_profile(sim)
    out["recommend_kernel_ms"] = kernel_profile(rec)
    return out


def catalogue(core, K: int, reps: int) -> dict:
    tr = model(core, 1, C1_ITEMS, K, seed=K)
    flop = 2.0 * C1_ITEMS * C1_ITEMS * K
    sim = lambda: tr.similar(1, None, C1_CUTOFF)  # noqa: E731
    sim()
    return {"items": C1_ITEMS, "K": K, "cutoff": C1_CUTOFF, "metric": "cosine",
            "similar_all_items": stats([timed(sim) for _ in range(reps)], flop)}


def _rank(rank: int, world: int, reps: int, barrier, q) -> None:
    import torch

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import balanced_bounds

    torch.cuda.set_device(rank)
    os.environ["IALS_B200_DEVICE"] = str(rank)
    tr = model(core, 1, BIG_ITEMS, BIG_K, seed=11)
    b = balanced_bounds(np.ones(BIG_ITEMS), world)
    sim = lambda: tr.similar(1, range(int(b[rank]), int(b[rank + 1])), BIG_CUTOFF)  # noqa: E731
    sim()
    times = []
    for _ in range(reps):
        barrier.wait()
        times.append(timed(sim))
    q.put((rank, times, card(rank)))


def multi_gpu(world: int, reps: int) -> dict:
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    barrier, q = ctx.Barrier(world), ctx.Queue()
    procs = [ctx.Process(target=_rank, args=(r, world, reps, barrier, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=1800) for _ in procs)
    for p in procs:
        p.join()
    per_pass = np.max(np.array([t for _, t, _ in got]), axis=0)
    flop = 2.0 * BIG_ITEMS * BIG_ITEMS * BIG_K
    return {"gpus": world, "items": BIG_ITEMS, "K": BIG_K, "cutoff": BIG_CUTOFF,
            "similar_all_items": stats(list(per_pass), flop), "cards": [c for _, _, c in got]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03d_similar.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("time_similar.py measures on a GPU; none is visible")
    from irspack_b200 import _ials_core as core

    result = {"card": card(0), "reps": a.reps}
    result["c1_k128"] = catalogue(core, 128, max(a.reps, 10))
    print(json.dumps(result["c1_k128"]), flush=True)
    result["c1_k256"] = catalogue(core, 256, max(a.reps, 10))
    print(json.dumps(result["c1_k256"]), flush=True)
    result["graph_2M"] = big_graph(core, a.reps)
    print(json.dumps(result["graph_2M"]), flush=True)
    result["multi_gpu"] = multi_gpu(a.gpus, a.reps) if a.gpus > 1 else "not measured (one GPU)"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
