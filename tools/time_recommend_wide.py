#!/usr/bin/env python
"""Times recommendation lists of a wide model (row stride > 128) on the configs[2] shape.

    python tools/time_recommend_wide.py --baseline-repo ../base [--out result.json]

configs[2] is 480 189 users x 17 770 items (the Netflix shape) with a synthetic power-law
training matrix of 100 480 507 entries (``dist.synth_user_block_device``, the device twin of
``synth.synth_csr``; the host generator takes minutes at this size) as the mask, and random
factors at K = 256 and 512.  Patterns, all top-10:

* ``all users, mask=train``: one ``IALSTrainer.recommend`` call over every user.  This tree runs
  the fused tcgen05 kernel at these strides; ``--baseline-repo`` (a checkout of the commit to
  compare with, built in place: ``git worktree add ../base <rev>`` and ``__graft_entry__.build()``
  there) runs whatever that commit runs -- before the wide kernel, the FP32 SIMT route of score.cu
  (score block in HBM, scatter mask, top-k).  The two run in separate worker processes and are
  timed alternately, after a warm-up call each; the lists of the two are compared.
* ``32 768 users, per-user allow-lists``: fused in one call, against the host fallback the
  Evaluator takes where the fused kernel does not apply (``user_scores`` score block to the host,
  then ``select_topk`` with the mask and the lists).

Times are host wall clock around a synchronous call (the lists are copied back inside it), the
median and the minimum of ``--reps`` repeats; the algorithmic rate is 2 U I K / t.  The card's name
and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

N_USERS, N_ITEMS, NNZ = 480_189, 17_770, 100_480_507
K_LIST = (256, 512)
CUTOFF = 10
ALLOW_USERS = 32_768


# ------------------------------------------------------------------ worker (one code tree) ----
def worker(repo: str) -> None:
    """Reads commands from stdin, answers one JSON line each.  Imports the package of ``repo``."""
    sys.path.insert(0, os.path.abspath(repo))
    import torch

    from irspack_b200 import _ials_core as core
    from irspack_b200.dist import synth_user_block_device
    from irspack_b200.evaluation import select_topk
    import scipy.sparse as sps

    dev = torch.device("cuda", 0)
    ip, ix, dt = synth_user_block_device(N_USERS, N_ITEMS, NNZ, seed=1002, device=dev, item_seed=7)
    X = sps.csr_matrix((dt.cpu().numpy(), ix.cpu().numpy(), ip.cpu().numpy()), shape=(N_USERS, N_ITEMS))
    del ip, ix, dt
    torch.cuda.empty_cache()
    rng = np.random.default_rng(3)
    lens = rng.integers(0, 1000, size=ALLOW_USERS)
    a_ip = np.zeros(ALLOW_USERS + 1, np.int64)
    np.cumsum(lens, out=a_ip[1:])
    a_ix = np.concatenate([np.sort(rng.choice(N_ITEMS, int(c), replace=False)) for c in lens]).astype(np.int32)
    allowed = (ALLOW_USERS, a_ip, a_ix)
    allowed_host = (ALLOW_USERS, a_ip, a_ix.astype(np.int64))  # the Evaluator's host form: int64 ids
    t = None
    sc = core.IALSSolverConfigBuilder().build()
    print(json.dumps({"ready": True, "nnz": int(X.nnz), "indices_sum": int(X.indices.sum(dtype=np.int64))}),
          flush=True)
    for line in sys.stdin:
        cmd = json.loads(line)
        op = cmd["op"]
        if op == "model":
            K = cmd["K"]
            t = None
            cfg = core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(1e-3).build()
            t = core.IALSTrainer(cfg, X)
            r = np.random.default_rng(K)
            user = (0.1 * r.standard_normal((N_USERS, K))).astype(np.float32)
            item = (0.1 * r.standard_normal((N_ITEMS, K))).astype(np.float32)
            t.user, t.item = user, item
            out = {"K": K}
        elif op == "ties":
            # rows whose lists differ between two runs: the largest float64 score gap between items
            # that traded places, over the row's largest |score| (a float32 near-tie is ~1e-6)
            a, b = np.load(cmd["a"]), np.load(cmd["b"])
            worst = 0.0
            for row in np.flatnonzero((a != b).any(axis=1)):
                s64 = user[row].astype(np.float64) @ item.astype(np.float64).T
                s64[X.indices[X.indptr[row]: X.indptr[row + 1]]] = -np.inf
                scale = np.abs(s64[np.isfinite(s64)]).max()
                for i, j in zip(a[row], b[row]):
                    if i != j:
                        worst = max(worst, abs(s64[i] - s64[j]) / scale)
            out = {"max_rel_score_gap_of_swaps": worst}
        elif op == "all":
            t0 = time.perf_counter()
            idx, cnt = t.recommend(0, N_USERS, CUTOFF, mask="train")
            out = {"ms": 1e3 * (time.perf_counter() - t0)}
            if cmd.get("dump"):
                np.save(cmd["dump"], idx)
        elif op == "allow_fused":
            t0 = time.perf_counter()
            idx, cnt = t.recommend(0, ALLOW_USERS, CUTOFF, mask="train", allowed=allowed)
            out = {"ms": 1e3 * (time.perf_counter() - t0)}
            if cmd.get("dump"):
                np.save(cmd["dump"], idx)
        elif op == "allow_host":
            t0 = time.perf_counter()
            scores = t.user_scores(0, ALLOW_USERS, sc)
            idx, cnt = select_topk(scores, CUTOFF, X[:ALLOW_USERS], allowed_host)
            out = {"ms": 1e3 * (time.perf_counter() - t0)}
            del scores
            if cmd.get("dump"):
                np.save(cmd["dump"], idx)
        else:
            raise ValueError(op)
        print(json.dumps(out), flush=True)


# ------------------------------------------------------------------------------- driver ----
class Worker:
    def __init__(self, repo: str):
        self.p = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", repo],
                                  stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True)
        self.info = self._read()

    def _read(self) -> dict:
        line = self.p.stdout.readline()
        if not line:
            raise RuntimeError(f"worker exited with {self.p.wait()}")
        return json.loads(line)

    def __call__(self, **cmd) -> dict:
        self.p.stdin.write(json.dumps(cmd) + "\n")
        self.p.stdin.flush()
        return self._read()

    def close(self) -> None:
        self.p.stdin.close()
        self.p.wait()


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def stats(ms) -> dict:
    return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "ms": [round(x, 3) for x in ms]}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--baseline-repo", required=False, default=None,
                    help="built checkout of the commit to compare with")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--tmp", default="/tmp")
    a = ap.parse_args()
    if a.worker:
        worker(a.worker)
        return
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    result = {"shape": {"users": N_USERS, "items": N_ITEMS, "mask_nnz": NNZ, "cutoff": CUTOFF},
              "card": card(), "reps": a.reps, "runs": []}
    new = Worker(here)
    base = Worker(a.baseline_repo) if a.baseline_repo else None
    result["mask_check"] = {"new": new.info, "baseline": base.info if base else None}
    for K in K_LIST:
        flop = 2.0 * N_USERS * N_ITEMS * K
        for w in (new, base):
            if w:
                w(op="model", K=K)
        fn = {w: os.path.join(a.tmp, f"rec_{K}_{name}.npy") for w, name in ((new, "new"), (base, "base")) if w}
        for w in fn:  # warm-up (scratch buffers, the sortedness check of the mask) + the lists
            w(op="all", dump=fn[w])
        times = {w: [] for w in fn}
        for _ in range(a.reps):
            for w in fn:
                times[w].append(w(op="all")["ms"])
        run = {"K": K, "pattern": f"all users, top-{CUTOFF}, mask=train"}
        for w, name in ((new, "fused (this tree)"), (base, "baseline")):
            if w:
                s = stats(times[w])
                s["tflops_algorithmic"] = flop / (s["median_ms"] * 1e-3) / 1e12
                run[name] = s
        if base:
            x, y = np.load(fn[new]), np.load(fn[base])
            run["rows_whose_lists_differ"] = int((x != y).any(axis=1).sum())
            run.update(new(op="ties", a=fn[new], b=fn[base]))
        result["runs"].append(run)
        print(json.dumps(run), flush=True)
        # per-user allow-lists: fused against the Evaluator's host fallback, both in this tree
        flop_a = 2.0 * ALLOW_USERS * N_ITEMS * K
        fa, fh = os.path.join(a.tmp, f"allow_{K}_fused.npy"), os.path.join(a.tmp, f"allow_{K}_host.npy")
        new(op="allow_fused", dump=fa)
        new(op="allow_host", dump=fh)
        tf, th = [], []
        for _ in range(a.reps):
            tf.append(new(op="allow_fused")["ms"])
            th.append(new(op="allow_host")["ms"])
        run = {"K": K, "pattern": f"{ALLOW_USERS} users, per-user allow-lists, top-{CUTOFF}, mask=train",
               "allowed_entries_per_user": "uniform 0..999"}
        for name, ms in (("fused (this tree)", tf), ("host score block + select_topk", th)):
            s = stats(ms)
            s["tflops_algorithmic"] = flop_a / (s["median_ms"] * 1e-3) / 1e12
            run[name] = s
        run["rows_whose_lists_differ"] = int((np.load(fa) != np.load(fh)).any(axis=1).sum())
        run.update(new(op="ties", a=fa, b=fh))
        result["runs"].append(run)
        print(json.dumps(run), flush=True)
    result["card_after"] = card()
    new.close()
    if base:
        base.close()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
