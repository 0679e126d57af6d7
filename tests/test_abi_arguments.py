"""Argument validation of the C ABI for malformed host inputs: each call runs in a subprocess, so an
input the library dereferences without checking shows up as a dead process rather than a dead suite."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# ials_topk_scores on 2 rows x 4 items, k = 1, with the mask given as (indptr, indices)
TOPK_CALL = r"""
import ctypes, sys
sys.path.insert(0, {root!r})
from irspack_b200 import _lib
P = ctypes.c_void_p
def arr(ctype, values):
    return None if values is None else (ctype * len(values))(*values)
scores = arr(ctypes.c_float, [0.1, 0.4, 0.3, 0.2, 0.9, 0.8, 0.7, 0.6])
indptr, indices = arr(ctypes.c_int64, {indptr!r}), arr(ctypes.c_int32, {indices!r})
idx, sc, cnt = arr(ctypes.c_int32, [0, 0]), arr(ctypes.c_float, [0, 0]), arr(ctypes.c_int32, [0, 0])
ptr = lambda a: None if a is None else ctypes.cast(a, P)
st = _lib.lib.ials_topk_scores(ptr(scores), 2, 4, 1, ptr(indptr), ptr(indices), 0, None, ptr(idx), ptr(sc),
                               ptr(cnt))
print(st, (_lib.lib.ials_last_error() or b"").decode() if st else "")
"""

IALS_OK, IALS_ERR_INVALID_ARGUMENT, IALS_ERR_CUDA = 0, 1, 3


def run_topk(indptr, indices):
    res = subprocess.run([sys.executable, "-c", TOPK_CALL.format(root=ROOT, indptr=indptr, indices=indices)],
                         capture_output=True, text=True, cwd=ROOT, timeout=300)
    assert res.returncode == 0, f"process died (rc {res.returncode}): {res.stderr[-2000:]}"
    status, _, message = res.stdout.strip().partition(" ")
    return int(status), message


@pytest.mark.parametrize("indptr, indices", [
    (None, [1, 2]),    # indices without indptr
    ([0, 1, 2], None),  # entries without indices
])
def test_topk_scores_rejects_malformed_mask(indptr, indices):
    status, message = run_topk(indptr, indices)
    assert status == IALS_ERR_INVALID_ARGUMENT, message
    assert "mask indptr / indices must both be given" in message


@pytest.mark.parametrize("indptr, indices", [
    (None, None),       # no mask
    ([0, 1, 2], [1, 2]),  # a mask with entries
    ([0, 0, 0], None),  # an empty mask needs no indices
])
def test_topk_scores_accepts_mask(indptr, indices):
    status, message = run_topk(indptr, indices)
    from irspack_b200 import _lib
    if _lib.device_count() == 0:  # past argument validation: no CPU fallback
        assert status == IALS_ERR_CUDA and "no CPU fallback" in message, message
    else:
        assert status == IALS_OK, message
