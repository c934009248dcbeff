"""CPU restatement of the RSA resampling entries of include/hba.h (hba_rank_order_f64, hba_rsa_perm_null,
hba_rsa_bootstrap and their workspace queries), by the formulas written in the header - test infrastructure only.

Importing this module attaches the entries to oracle.libhba_ref.RefLib, so that `emulated_device()` serves them like
every other entry point: the host side of hba.rsa's permutation_test / bootstrap then runs unmodified on CPU tensors,
and tests/emulate_clip_gpu_tests.py can dry-run tests/test_gpu_rsa_stats.py.  The argument checks of the front ends
are restated (HBA_ERR_ARG and a message in hba_last_error()).

The bootstrap is restated the way the kernels compute it - weighted average ranks over the fixed sorted order - and
tests/test_rsa_stats_cpu.py shows that this equals scipy.stats.rankdata on the explicitly expanded multiset.
"""
import numpy as np
import torch

from oracle import libhba_ref
from oracle.libhba_ref import _addr, _al, _require, flat

MAX_N = 2191   # exact int64 sums: 2 P^3 / 3 < 2^63


def sorted_order(x):
    """(stable sorted order, keys) of float64 values under the library's key order: -0.0 == +0.0, NaN with the sign
    bit clear above +inf, NaN with it set below -inf."""
    bits = (np.asarray(x, dtype=np.float64) + 0.0).view(np.uint64)
    neg = (bits >> np.uint64(63)).astype(bool)
    keys = np.where(neg, ~bits, bits | np.uint64(1 << 63))
    return np.argsort(keys, kind="stable"), keys


def perm_null_ref(ref_ranks, model_ranks, N, perms):
    """rho_p = Pearson over i<j of (ref_ranks[i,j], model_ranks[pi_p(i), pi_p(j)]); NaN for NaN ranks, for a constant
    side or for an entry of pi_p outside [0, N)."""
    out = np.full(len(perms), np.nan)
    if np.isnan(ref_ranks).any() or np.isnan(model_ranks).any():
        return out
    i, j = np.triu_indices(N, k=1)
    Bm = np.zeros((N, N))
    Bm[i, j] = Bm[j, i] = model_ranks
    for p, pi in enumerate(perms):
        if pi.min() < 0 or pi.max() >= N:
            continue
        with np.errstate(all="ignore"):
            out[p] = np.clip(np.corrcoef(ref_ranks, Bm[pi[i], pi[j]])[0, 1], -1.0, 1.0)
    return out


def weighted_average_ranks(x, order, w):
    """Average ranks, in pair order, of the multiset in which entry k of x appears w[k] times, scanned in the fixed
    sorted order `order` of x: a tie group g of total weight W_g after groups of total weight S_g has the rank
    S_g + (W_g + 1) / 2.  Entries of weight 0 get the rank of their group, which no weighted sum sees."""
    keys = sorted_order(x)[1][order]
    ws = np.asarray(w, dtype=np.int64)[order]
    start = np.ones(len(keys), dtype=bool)
    start[1:] = keys[1:] != keys[:-1]
    gid = np.cumsum(start) - 1
    W = np.bincount(gid, weights=ws, minlength=gid[-1] + 1).astype(np.int64)
    S = np.concatenate([[0], np.cumsum(W)[:-1]])
    r = np.empty(len(x))
    r[order] = S[gid] + (W[gid] + 1) / 2.0
    return r


def bootstrap_rho_ref(ref, model, N, counts):
    """rho of one stimulus-bootstrap replicate: pairs {i,j}, i != j, weighted by counts[i] counts[j], weighted Pearson
    of the weighted average ranks; NaN when the counts are not N values in [0, N] summing to N, when a pair of weight
    > 0 is NaN in either RDM or when a side is constant.  ref, model: (upper triangle, its sorted order)."""
    c = np.asarray(counts, dtype=np.int64)
    if c.min() < 0 or c.max() > N or c.sum() != N:
        return np.nan
    i, j = np.triu_indices(N, k=1)
    w = c[i] * c[j]
    live = w > 0
    (xr, o_r), (xm, o_m) = ref, model
    if np.isnan(xr[live]).any() or np.isnan(xm[live]).any():
        return np.nan
    M = w.sum()
    a = 2 * weighted_average_ranks(xr, o_r, w) - (M + 1)
    b = 2 * weighted_average_ranks(xm, o_m, w) - (M + 1)
    saa, sbb, sab = (w * a * a)[live].sum(), (w * b * b)[live].sum(), (w * a * b)[live].sum()
    if saa <= 0 or sbb <= 0:
        return np.nan
    return float(np.clip(sab / np.sqrt(saa) / np.sqrt(sbb), -1.0, 1.0))


# ---------------------------------------------------------------- the entry points, as RefLib methods
def hba_rank_order_f64(self, x, n, order, ranks, workspace, workspace_bytes, stream):
    from scipy.stats import rankdata
    _require(_addr(x) and _addr(order) and _addr(ranks) and n > 0, "bad arguments")
    xv = flat(x, n, torch.float64).numpy()
    flat(order, n, torch.int32).copy_(torch.from_numpy(sorted_order(xv)[0].astype(np.int32)))
    flat(ranks, n, torch.float64).copy_(torch.from_numpy(rankdata(xv, nan_policy="propagate")))
    return self._ok("hba_rank_order_f64")


def hba_rsa_perm_workspace_bytes(self, N, n_perm):
    return 0 if N < 2 or n_perm < 1 else 8 * N * N + 16 * n_perm + 512


def hba_rsa_perm_null(self, ref_ranks, model_ranks, N, perms, n_perm, rho_out, workspace, workspace_bytes, stream):
    _require(_addr(ref_ranks) and _addr(model_ranks) and _addr(perms) and _addr(rho_out), "null pointer")
    _require(3 <= N <= MAX_N, f"N={N} outside [3, {MAX_N}] (exact int64 sums)")
    _require(1 <= n_perm <= 65535 * 8, f"n_perm={n_perm} outside [1, {65535 * 8}]")
    _require(_al(perms, 4) and _al(ref_ranks, 8) and _al(model_ranks, 8) and _al(rho_out, 8), "misaligned pointer")
    # (the library also needs 256-byte alignment, which CUDA allocations give; host tensors are only 64-byte aligned)
    _require(_addr(workspace) and workspace_bytes >= hba_rsa_perm_workspace_bytes(self, N, n_perm),
             "workspace too small")
    P = N * (N - 1) // 2
    pi = flat(perms, n_perm * N, torch.int32).view(n_perm, N).numpy()
    flat(rho_out, n_perm, torch.float64).copy_(torch.from_numpy(perm_null_ref(
        flat(ref_ranks, P, torch.float64).numpy(), flat(model_ranks, P, torch.float64).numpy(), N, pi)))
    return self._ok("hba_rsa_perm_null")


def hba_rsa_boot_workspace_bytes(self, N, n_boot):
    P = N * (N - 1) // 2
    return 0 if N < 2 or n_boot < 1 else 44 * P + n_boot * (8 * P + 64) + 4096


def hba_rsa_bootstrap(self, ref_tri, ref_order, tri_a, order_a, tri_b, order_b, N, counts, n_boot, rho_a, rho_b,
                      workspace, workspace_bytes, stream):
    _require(_addr(ref_tri) and _addr(ref_order) and _addr(tri_a) and _addr(order_a) and _addr(counts)
             and _addr(rho_a), "null pointer")
    _require((_addr(tri_b) == 0) == (_addr(order_b) == 0) == (_addr(rho_b) == 0),
             "tri_b, order_b and rho_b are given together or not at all")
    _require(3 <= N <= MAX_N, f"N={N} outside [3, {MAX_N}] (exact int64 sums)")
    _require(1 <= n_boot <= 65535, f"n_boot={n_boot} outside [1, 65535]")
    _require(all(_al(t, 8) for t in (ref_tri, tri_a, tri_b, rho_a, rho_b))
             and all(_al(t, 4) for t in (ref_order, order_a, order_b, counts)), "misaligned pointer")
    _require(_addr(workspace) and workspace_bytes >= hba_rsa_boot_workspace_bytes(self, N, n_boot),
             "workspace too small")
    P = N * (N - 1) // 2
    c = flat(counts, n_boot * N, torch.int32).view(n_boot, N).numpy()
    vec = lambda t, o: (flat(t, P, torch.float64).numpy(), flat(o, P, torch.int32).numpy().view(np.uint32))
    ref = vec(ref_tri, ref_order)
    models = [(vec(tri_a, order_a), rho_a)] + ([(vec(tri_b, order_b), rho_b)] if _addr(tri_b) else [])
    for (x, order), out in models:
        flat(out, n_boot, torch.float64).copy_(torch.from_numpy(
            np.array([bootstrap_rho_ref(ref, (x, order), N, cb) for cb in c], dtype=np.float64)))
    return self._ok("hba_rsa_bootstrap")


ENTRIES = (hba_rank_order_f64, hba_rsa_perm_workspace_bytes, hba_rsa_perm_null, hba_rsa_boot_workspace_bytes,
           hba_rsa_bootstrap)
for _fn in ENTRIES:
    setattr(libhba_ref.RefLib, _fn.__name__, _fn)
del _fn
