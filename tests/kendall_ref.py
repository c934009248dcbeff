"""CPU restatement of hba_kendall_tau_f64 and hba_kendall_workspace_bytes (include/hba.h) by the header's formulas, and
an independent exact oracle of the pair counts - test infrastructure only.

Importing this module attaches the entries to oracle.libhba_ref.RefLib, so that `emulated_device()` serves them like
every other entry point: RSAEvaluator.kendall_tau and hba.rsa_scale then run unmodified on CPU tensors, and
tests/emulate_clip_gpu_tests.py can dry-run tests/test_gpu_kendall.py.  The argument checks of the front end are
restated (HBA_ERR_ARG and a message in hba_last_error()).

The oracle shares nothing with the kernels' algorithm beyond the definitions: ties are counted with numpy.unique, and
the discordant pairs are the strict inversions of y's dense ranks in (x, y) lexicographic order, counted by a bottom-up
merge in which every level is one vectorised numpy.searchsorted over all pairs of runs, O(n log n) in all.
"""
import numpy as np
import torch

import rsa_stats_ref  # noqa: F401  (hba_rank_order_f64 on the restatement: RSAEvaluator sorts the reference with it)
from oracle import libhba_ref
from oracle.libhba_ref import _addr, _al, _require, flat

SMALL_N = 2048     # one CTA up to here; larger n needs the workspace
MAX_N = 1 << 30    # exclusive, the bound of hba_rank_order_f64


def _tie_pairs(v):
    """sum t(t-1)/2 over the groups of equal values (rows of a 2-D array) of v."""
    t = np.unique(v, axis=0, return_counts=True)[1].astype(np.int64)
    return int((t * (t - 1) // 2).sum())


def strict_inversions(a):
    """#{i < j : a[i] > a[j]} of non-negative integers a, by bottom-up merging: at width w the runs [s, s+w) and
    [s+w, s+2w) are sorted; every right-run element counts the left-run elements greater than it with one searchsorted
    over all left runs at once (values offset by run-pair index * (max + 1) keep the pairs apart), then the pairs are
    merged by the positions the same searches give."""
    a = np.asarray(a, dtype=np.int64).copy()
    n = len(a)
    span = int(a.max(initial=0)) + 1
    idx = np.arange(n)
    total, w = 0, 1
    while w < n:
        pair, off = idx // (2 * w), idx % (2 * w)
        left = off < w
        key = pair * span + a                  # sorted inside each run; runs of different pairs apart
        lk, rk = key[left], key[~left]         # all left runs concatenated, all right runs concatenated
        lpair, rpair = pair[left], pair[~left]
        lstart = np.searchsorted(lpair, rpair, "left")          # first left element of each right element's pair
        lend = np.searchsorted(lpair, rpair, "right")
        le = np.searchsorted(lk, rk, "right") - lstart          # left elements <= it (ties are not inversions)
        total += int(((lend - lstart) - le).sum())
        rstart = np.searchsorted(rpair, lpair, "left")
        lt = np.searchsorted(rk, lk, "left") - rstart           # right elements < a left element: it stays first
        out = np.empty_like(a)
        start = pair * 2 * w
        out[start[left] + off[left] + lt] = a[left]
        out[start[~left] + (off[~left] - w) + le] = a[~left]
        a, w = out, 2 * w
    return total


def kendall_counts(x, y):
    """(S, n1, n2, n3) of the header: exact Python ints, -0.0 == +0.0; None when x or y holds a NaN."""
    x = np.asarray(x, dtype=np.float64) + 0.0
    y = np.asarray(y, dtype=np.float64) + 0.0
    if np.isnan(x).any() or np.isnan(y).any():
        return None
    n = len(x)
    n0 = n * (n - 1) // 2
    n1, n2, n3 = _tie_pairs(x), _tie_pairs(y), _tie_pairs(np.stack([x, y], 1))
    o = np.lexsort((y, x))                                   # by x, ties in x by y: those pairs are never inversions
    yd = np.unique(y, return_inverse=True)[1].reshape(-1)
    D = strict_inversions(yd[o])
    return n0 - n1 - n2 + n3 - 2 * D, n1, n2, n3


def kendall_taus(counts, n):
    """(tau_a, tau_b) from the counts by the header's formulas (tau_b in scipy.stats.kendalltau's order of operations)."""
    if counts is None:
        return float("nan"), float("nan")
    S, n1, n2, _ = counts
    n0 = n * (n - 1) // 2
    if n1 == n0 or n2 == n0:
        return float("nan"), float("nan")
    tau_b = float(S) / np.sqrt(float(n0 - n1)) / np.sqrt(float(n0 - n2))
    return float(S) / float(n0), float(min(1.0, max(-1.0, tau_b)))


# ---------------------------------------------------------------- the entry points, as RefLib methods
def hba_kendall_workspace_bytes(self, n):
    return 256 if n <= SMALL_N else 44 * int(n) + (1 << 20)


def hba_kendall_tau_f64(self, x, y, y_order, n, counts, tau, workspace, workspace_bytes, stream):
    _require(_addr(x) and _addr(y) and _addr(y_order) and _addr(counts) and _addr(tau), "null pointer")
    _require(2 <= n < MAX_N, f"n={n} outside [2, 2^30)")
    _require(_al(x, 8) and _al(y, 8) and _al(y_order, 4) and _al(counts, 8) and _al(tau, 8), "misaligned pointer")
    if n > SMALL_N:
        # (the library also needs 256-byte alignment, which CUDA allocations give; host tensors are only 64-byte aligned)
        _require(_addr(workspace) and workspace_bytes >= hba_kendall_workspace_bytes(self, n), "workspace too small")
    xv, yv = flat(x, n, torch.float64).numpy(), flat(y, n, torch.float64).numpy()
    order = flat(y_order, n, torch.int32).numpy().view(np.uint32).astype(np.int64)
    keys = rsa_stats_ref.sorted_order(yv)[1]
    in_range = bool(order.max() < n)
    sorts_y = in_range and bool((keys[order][1:] >= keys[order][:-1]).all())
    c = kendall_counts(xv, yv) if sorts_y else None
    flat(counts, 4, torch.int64).copy_(torch.tensor(c if c is not None else (-1, -1, -1, -1), dtype=torch.int64))
    flat(tau, 2, torch.float64).copy_(torch.tensor(kendall_taus(c, n), dtype=torch.float64))
    return self._ok("hba_kendall_tau_f64")


ENTRIES = (hba_kendall_workspace_bytes, hba_kendall_tau_f64)
for _fn in ENTRIES:
    setattr(libhba_ref.RefLib, _fn.__name__, _fn)
del _fn
