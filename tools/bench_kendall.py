#!/usr/bin/env python
"""Time per call of Kendall's tau on the GPU (hba_kendall_tau_f64) against scipy.stats.kendalltau on the host, at the
per-epoch RSA size (N = 48 images, P = 1,128 pairs) and at RSA at scale (N = 1,854, P = 1,717,731):

    python tools/bench_kendall.py [--sizes 48 1854] [--min-seconds 1.0] [--out result.json]

For each N: the time per call from CUDA events over a window of at least --min-seconds after a warm-up call of the same
shape (model triangle of random 66-D embeddings against a reference RDM, the reference's sorted order given, as
RSAEvaluator.kendall_tau calls it); the kernel time of each phase from torch.profiler in a separate run, the bytes each
phase moves by the algorithm (computed from P, not measured) and the bandwidth that gives; scipy's time per call on
this host's CPU and whether the values agree; the card's name and power limit, read in the same run.  The working set
(about 70 bytes per pair, 120 MB at N = 1,854) stays in the 126 MB L2 from call to call.  Prints one JSON line.
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


def _executed_digit_passes(x_perm):
    """Digit passes the radix sort runs on the keys of x[y_order]: those whose byte is not the same for every key."""
    import numpy as np
    bits = (np.asarray(x_perm, dtype=np.float64) + 0.0).view(np.uint64)
    neg = (bits >> np.uint64(63)).astype(bool)
    keys = np.where(neg, ~bits, bits | np.uint64(1 << 63))
    return sum(int(len(np.unique((keys >> np.uint64(8 * d)) & np.uint64(255))) > 1) for d in range(8))


def phase_bytes(P, passes):
    """Bytes each phase reads and writes by the algorithm (4-byte indices, 8-byte keys and values; gathers counted at
    their element size, not their 32-byte sectors)."""
    levels, w = 0, 4096
    while w < P:
        levels, w = levels + 1, 2 * w
    if P <= 2048:
        return {"one_cta": 4 * P + 16 * P + 48}, 0
    return {
        "keys": 4 * P + 4 * P + 16 * P + 8 * P + 8 * P,          # y_order (twice), x and y gathered, ky and keys written
        "radix_sort": 8 * P + passes * 24 * P,                   # histogram pass, then keys + indices in and out
        "ranks": 8 * P + 4 * P + 8 * P + 4 * P,                  # ky, sorted indices, ky at them, y-ranks written
        "tile": 4 * P + 8 * P + 4 * P,                           # y-ranks and sorted keys read, sorted tiles written
        "merge_levels": levels * 8 * P,                          # every level reads and writes the y-ranks once
    }, levels


PHASE_OF = {"kendall_small_kernel": "one_cta", "kendall_keys_kernel": "keys", "radix_hist_kernel": "radix_sort",
            "radix_pass_kernel": "radix_sort", "kendall_ranks_kernel": "ranks", "kendall_tile_kernel": "tile",
            "kendall_merge_kernel": "merge_levels", "kendall_final_kernel": "final"}


def _phase_times(fn, calls=20):
    """Kernel time per call of each phase (torch.profiler, CUDA activities), in a run of its own."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        for kname, phase in PHASE_OF.items():
            if kname in ev.key:
                out[phase] = out.get(phase, 0.0) + ev.device_time_total / 1e6 / calls
    return out


def bench(N, min_seconds, host_reps):
    import numpy as np
    import torch
    from hba import ops
    from hba.rsa import RSAEvaluator
    from scipy.stats import kendalltau
    rng = np.random.default_rng(N)
    ref = 1 - np.corrcoef(rng.standard_normal((N, 66)))
    np.fill_diagonal(ref, 0)
    emb = torch.from_numpy(rng.standard_normal((N, 66)).astype(np.float32)).cuda()
    ev = RSAEvaluator(ref, "cuda")
    P = ev.P
    x = torch.empty(P, dtype=torch.float64, device="cuda")
    ops.rdm_f64(emb, None, x)
    order = ev._reference_order()
    counts = torch.empty(4, dtype=torch.int64, device="cuda")
    tau = torch.empty(2, dtype=torch.float64, device="cuda")
    ws = torch.empty(ops.kendall_workspace_bytes(P), dtype=torch.uint8, device="cuda")
    call = lambda: ops.kendall_tau_f64(x, ev.ref_tri, order, counts, tau, ws)
    per_call, calls = _timed(call, min_seconds)
    phases = _phase_times(call)
    xh, yh = x.cpu().numpy(), ev.ref_tri.cpu().numpy()
    host = []
    for _ in range(host_reps):
        t0 = time.perf_counter()
        want = float(kendalltau(xh, yh).statistic)
        host.append(time.perf_counter() - t0)
    got = tau.cpu().tolist()
    passes = _executed_digit_passes(xh[order.cpu().numpy().view(np.uint32)])
    nbytes, levels = phase_bytes(P, passes)
    return {
        "N": N, "pairs": P, "calls_timed": calls, "window_s": per_call * calls, "s_per_call": per_call,
        "kernels_per_call": ops.kendall_kernels(P), "radix_digit_passes_executed": passes, "merge_levels": levels,
        "phases": {ph: {"kernel_s_per_call": phases.get(ph), "bytes": b,
                        "bytes_per_s": b / phases[ph] if phases.get(ph) else None,
                        "fraction_of_hbm_bandwidth": b / phases[ph] / HBM_BYTES_PER_S if phases.get(ph) else None}
                   for ph, b in nbytes.items()},
        "final_kernel_s_per_call": phases.get("final"),
        "kernel_s_per_call_sum": sum(phases.values()),
        "scipy_host_s_per_call": min(host), "scipy_host_s_all": host, "speedup_vs_scipy": min(host) / per_call,
        "tau_a": got[0], "tau_b": got[1], "tau_b_equals_scipy": got[1] == want,
        "goal_2ms_met": per_call < 2e-3 if N == 1854 else None,
    }


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", type=int, nargs="+", default=[48, 1854])
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--host-reps", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args(argv)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_kendall needs a CUDA device")
    res = {"metric": "Kendall's tau-a / tau-b of one RDM against a reference: seconds per call", "card": _card(),
           "host_cpus": os.cpu_count(), "sizes": [bench(N, a.min_seconds, a.host_reps) for N in a.sizes]}
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
