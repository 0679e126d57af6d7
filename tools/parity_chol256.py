#!/usr/bin/env python
"""Cholesky half-epochs at K in (224, 256] (row stride 256) against the oracle; prints one JSON
line with the errors.  The tensor-core route is the default; run under IALS_CHOL=simt to check the register-tiled kernel of
irspack_b200/csrc/solve.cu solve_cholesky_tensor (tests/test_zz_experimental.py does)."""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import oracle  # noqa: E402
from irspack_b200 import _ials_core as core  # noqa: E402
from irspack_b200.synth import init_factors, synth_csr  # noqa: E402

out = {"IALS_CHOL": os.environ.get("IALS_CHOL", "")}
for K, loss in ((256, "IALSPP"), (240, "ORIGINAL")):
    U, I, nnz = 600, 150, 30000  # items average 200 neighbours, the heaviest several hundred
    X = synth_csr(U, I, nnz, seed=21, values="counts")
    X = X.tolil()
    X[7, :] = 0  # a user without interactions
    X = X.tocsr()
    X.eliminate_zeros()
    u0, i0 = init_factors(U, K, 1), init_factors(I, K, 2)
    cfg = (core.IALSModelConfigBuilder().set_K(K).set_alpha0(0.1).set_reg(0.02)
           .set_loss_type(getattr(core.LossType, loss)).build())
    sc = core.IALSSolverConfigBuilder().set_solver_type(core.SolverType.CHOLESKY).build()
    g = core.IALSTrainer(cfg, X)
    g.user, g.item = u0, i0
    lt = oracle.LOSS_ORIGINAL if loss == "ORIGINAL" else oracle.LOSS_IALSPP
    o32 = oracle.OracleTrainer(X, K, 0.1, 0.02, 1.0, lt, dtype=np.float32)
    o64 = oracle.OracleTrainer(X, K, 0.1, 0.02, 1.0, lt, dtype=np.float64)
    for o in (o32, o64):
        o.user, o.item = u0.astype(o.dtype), i0.astype(o.dtype)
    errs = {}
    for side in (0, 1):
        g.half_step(side, sc)
        for o in (o32, o64):
            if side == 0:
                o._solve(o.user, o.X, o.item, oracle.SOLVER_CHOLESKY, 3, 2)
            else:
                o._solve(o.item, o.X_t, o.user, oracle.SOLVER_CHOLESKY, 3, 2)
        got = g.user if side == 0 else g.item
        w32, w64 = (o32.user, o64.user) if side == 0 else (o32.item, o64.item)
        scale = np.abs(w64).max()
        errs[f"side{side}_vs_f64"] = float(np.abs(got - w64).max() / scale)
        errs[f"side{side}_oracle32_vs_f64"] = float(np.abs(w32 - w64).max() / scale)
        if side == 0:
            errs["empty_row_is_zero"] = bool(not got[7].any())
    out[f"K{K}_{loss}"] = errs
print(json.dumps(out))
