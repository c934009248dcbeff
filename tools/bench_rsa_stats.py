#!/usr/bin/env python
"""Throughput of the RSA resampling statistics on the GPU (hba_rsa_perm_null, hba_rsa_bootstrap) against a host
evaluation, at the per-epoch RSA size (N = 48) and at RSA at scale (N = 1,854):

    python tools/bench_rsa_stats.py [--sizes 48 1854] [--min-seconds 1.0] [--out result.json]

For each N: permutations/s and bootstrap replicates/s (one model against the reference), timed with CUDA events over a
window of at least --min-seconds after a warm-up call of the same shape; the bytes and integer operations per
replicate that the kernels' algorithm needs (computed from N, not measured); the achieved rates and their fraction of
the HBM bandwidth; the L2 state (the working set of one call against the 126 MB L2); the time per replicate of the
same replicates evaluated on the host the way a reference RSA evaluation does it (RDMs indexed by the permutation or
resample, scipy.stats.spearmanr) and the largest difference from it; the card's name and power limit, read in the same
run.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vit-project_b200")]

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU
L2_BYTES = 126e6


def _card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip().splitlines()}


def _timed(fn, min_seconds):
    """(seconds per call, calls): CUDA events around repeated calls, the window grown to >= min_seconds."""
    import torch
    fn()
    torch.cuda.synchronize()
    calls = 1
    while True:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        e1.synchronize()
        s = e0.elapsed_time(e1) / 1e3
        if s >= min_seconds:
            return s / calls, calls
        calls = max(calls * 2, int(calls * min_seconds / max(s, 1e-6) * 1.2) + 1)


def perm_model(N, K=8):
    """Per permutation: row pi(i) of the model's N x N int32 rank matrix staged into shared memory for every row i
    (4 N^2 bytes, L2 -> SM), the reference rows read once per 8 permutations (4 N^2 / 8), the permutation itself
    (4 N); N^2 int32 x int32 -> int64 multiply-adds."""
    return {"bytes": 4 * N * N + 4 * N * N / K + 4 * N, "int_madds": N * N,
            "working_set_bytes": 8 * N * N}


def boot_model(N, reps):
    """Per replicate and RDM (reference, model): the weight prefix written and read (4 P + 4 P), the reference's
    ranks scattered to pair order / gathered by the model pass (4 P each, 32-byte sectors for 4-byte accesses), the
    per-position codes (pair, tie group bounds: 12 P per RDM) read by four kernels once per batch of 8 replicates;
    about 10 integer operations per pair and pass."""
    P = N * (N - 1) // 2
    logical = 2 * (4 * P + 4 * P) + 4 * P + 4 * P + 2 * 4 * 12 * P / 8
    sectors = logical - 8 * P + 2 * 32 * P
    return {"bytes": logical, "bytes_32B_sectors": sectors, "int_ops": 2 * 3 * 10 * P,
            "working_set_bytes": reps * 8 * P + 2 * 12 * P}


def bench(N, min_seconds, n_perm, n_boot, host_reps):
    import numpy as np
    import torch
    from hba import ops
    from hba.rsa import RSAEvaluator
    from scipy.stats import spearmanr
    rng = np.random.default_rng(N)
    t = rng.standard_normal((N, 66))
    ref = 1 - np.corrcoef(t)
    np.fill_diagonal(ref, 0)
    emb = torch.from_numpy(rng.standard_normal((N, 66)).astype(np.float32)).cuda()
    ev = RSAEvaluator(ref, "cuda")
    tri, order, ranks = ev._model_arrays(emb)
    ref_order = torch.empty_like(order)
    ops.rank_order_f64(ev.ref_tri, ref_order, torch.empty_like(ranks), ev.rank_ws)
    perms = torch.from_numpy(np.stack([rng.permutation(N) for _ in range(n_perm)]).astype(np.int32)).cuda()
    counts = torch.from_numpy(np.stack([np.bincount(rng.integers(0, N, N), minlength=N)
                                        for _ in range(n_boot)]).astype(np.int32)).cuda()
    rho_p = torch.empty(n_perm, dtype=torch.float64, device="cuda")
    rho_b = torch.empty(n_boot, dtype=torch.float64, device="cuda")
    ws_p = torch.empty(ops.rsa_perm_workspace_bytes(N, n_perm), dtype=torch.uint8, device="cuda")
    ws_b = torch.empty(ops.rsa_boot_workspace_bytes(N, n_boot), dtype=torch.uint8, device="cuda")
    sp, cp = _timed(lambda: ops.rsa_perm_null(ev.ref_ranks, ranks, perms, rho_p, ws_p), min_seconds)
    sb, cb = _timed(lambda: ops.rsa_bootstrap(ev.ref_tri, ref_order, tri, order, counts, rho_b, ws_b), min_seconds)
    # the same replicates evaluated on the host the way a reference RSA evaluation does it (this host's CPU): index
    # the two RDMs by the permutation / resample, drop the pairs of a stimulus with itself, scipy.stats.spearmanr
    iu = np.triu_indices(N, 1)
    R = np.zeros((N, N))
    R[iu] = ev.ref_tri.cpu().numpy()
    R += R.T
    m = np.zeros((N, N))
    m[iu] = tri.cpu().numpy()
    m += m.T
    t0 = time.perf_counter()
    host_null = np.array([spearmanr(R[iu], m[np.ix_(pi, pi)][iu])[0] for pi in perms[:host_reps].cpu().numpy()])
    t_host_perm = (time.perf_counter() - t0) / host_reps
    host_boot = []
    t0 = time.perf_counter()
    for c in counts[:host_reps].cpu().numpy():
        idx = np.repeat(np.arange(N), c)
        a, b = idx[iu[0]], idx[iu[1]]
        keep = a != b
        host_boot.append(spearmanr(R[a[keep], b[keep]], m[a[keep], b[keep]])[0])
    t_host_boot = (time.perf_counter() - t0) / host_reps
    host_boot = np.array(host_boot)
    dev_null, dev_boot = rho_p[:host_reps].cpu().numpy(), rho_b[:host_reps].cpu().numpy()
    pm, bm = perm_model(N), boot_model(N, n_boot)
    per_perm, per_boot = sp / n_perm, sb / n_boot
    return {
        "N": N, "pairs": N * (N - 1) // 2,
        "permutation": {
            "per_call": n_perm, "calls_timed": cp, "window_s": sp * cp, "perms_per_s": 1 / per_perm,
            "s_per_perm": per_perm, "model": pm, "bytes_per_s": pm["bytes"] / per_perm,
            "int_madds_per_s": pm["int_madds"] / per_perm,
            "fraction_of_hbm_bandwidth": pm["bytes"] / per_perm / HBM_BYTES_PER_S,
            "l2_state": ("warm: the call's working set (%.1f MB) fits the 126 MB L2 and is re-read by every call"
                         % (pm["working_set_bytes"] / 1e6)) if pm["working_set_bytes"] < L2_BYTES else
                        "working set exceeds L2",
            "host_s_per_perm": t_host_perm, "speedup_vs_host": t_host_perm / per_perm,
            "max_abs_diff_vs_host": float(np.nanmax(np.abs(dev_null - host_null))),
        },
        "bootstrap": {
            "per_call": n_boot, "calls_timed": cb, "window_s": sb * cb, "replicates_per_s": 1 / per_boot,
            "s_per_replicate": per_boot, "model": bm, "bytes_per_s": bm["bytes"] / per_boot,
            "sector_bytes_per_s": bm["bytes_32B_sectors"] / per_boot,
            "fraction_of_hbm_bandwidth": bm["bytes"] / per_boot / HBM_BYTES_PER_S,
            "l2_state": ("warm: the call's working set (%.1f MB) fits the 126 MB L2" % (bm["working_set_bytes"] / 1e6))
                        if bm["working_set_bytes"] < L2_BYTES else
                        "the call's working set (%.0f MB) exceeds the 126 MB L2: prefixes and ranks stream through HBM"
                        % (bm["working_set_bytes"] / 1e6),
            "host_s_per_replicate": t_host_boot, "speedup_vs_host": t_host_boot / per_boot,
            "max_abs_diff_vs_host": float(np.nanmax(np.abs(dev_boot - host_boot))),
        },
        "goal_10k_perm_plus_1k_boot_s": 10000 * per_perm + 1000 * per_boot,
    }


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[48, 1854])
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--host-reps", type=int, default=4)
    ap.add_argument("--out", default="")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_rsa_stats needs a CUDA device")
    res = {"metric": "RSA resampling statistics: permutations/s and bootstrap replicates/s", "card": _card(),
           "sizes": []}
    for N in a.sizes:
        n_perm, n_boot = (65536, 4096) if N <= 256 else (4096, 64)
        res["sizes"].append(bench(N, a.min_seconds, n_perm, n_boot, a.host_reps))
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
