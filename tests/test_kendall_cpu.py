"""Kendall's tau (hba.rsa.RSAEvaluator.kendall_tau, hba_kendall_tau_f64) on the CPU: the exact numpy oracle of
tests/kendall_ref.py against brute-force O(n^2) pair counting and against scipy.stats.kendalltau at the full RSA size,
the host API on the CPU restatement of libhba, the CSV columns of hba.rsa_scale and the tool's flag, and a dry run of
the GPU test file."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.stats import kendalltau

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from kendall_ref import kendall_counts, kendall_taus, strict_inversions  # noqa: E402


def _brute(x, y):
    """(S, n1, n2, n3) from every pair; -0.0 == +0.0 as numpy compares."""
    i, j = np.triu_indices(len(x), 1)
    sx, sy = np.sign(x[i] - x[j]), np.sign(y[i] - y[j])
    return (int((sx * sy).sum()), int((sx == 0).sum()), int((sy == 0).sum()), int(((sx == 0) & (sy == 0)).sum()))


@pytest.mark.parametrize("seed", range(8))
def test_oracle_equals_brute_force_with_heavy_ties(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(2, 700))
    levels = [2, 3, 7, 40, 10 ** 6][seed % 5]
    x = rng.integers(0, levels, n).astype(np.float64) - levels // 2
    y = rng.integers(0, [2, 5, 1000][seed % 3], n).astype(np.float64)
    x[x == 0] = np.where(rng.random((x == 0).sum()) < 0.5, -0.0, 0.0)
    assert kendall_counts(x, y) == _brute(x, y)


def test_strict_inversions_small_cases():
    assert strict_inversions([]) == 0 and strict_inversions([5]) == 0
    assert strict_inversions([3, 2, 1, 0]) == 6 and strict_inversions([1, 1, 1]) == 0
    a = np.random.default_rng(1).integers(0, 9, 301)
    assert strict_inversions(a) == sum(int((a[:k] > a[k]).sum()) for k in range(len(a)))


def test_oracle_tau_b_equals_scipy_at_the_full_rsa_size():
    """P = 1,717,731 pairs of a 1,854-image triangle, with ties on the reference side: tau_b == scipy's, exactly."""
    rng = np.random.default_rng(0)
    P = 1854 * 1853 // 2
    y = rng.integers(0, 40, P).astype(np.float64)
    x = y + rng.standard_normal(P) * 20
    c = kendall_counts(x, y)
    assert kendall_taus(c, P)[1] == float(kendalltau(x, y).statistic)
    assert kendall_taus(c, P)[0] == float(c[0]) / float(P * (P - 1) // 2)


def test_nan_and_constant_sides():
    x = np.arange(10.0)
    assert kendall_counts(np.where(x == 3, np.nan, x), x) is None
    assert all(np.isnan(kendall_taus(None, 10)))
    c = kendall_counts(np.ones(10), x)
    assert c == (0, 45, 0, 0) and all(np.isnan(kendall_taus(c, 10)))


@pytest.mark.parametrize("N", [48, 120])
def test_host_api_on_the_restatement(N):
    from hba.rsa import RSAEvaluator
    from oracle.libhba_ref import emulated_device
    from test_gpu_kendall import _data
    ref, emb = _data(N, seed=N)
    with emulated_device() as lib:
        ev = RSAEvaluator(ref, "cpu")
        tau_a, tau_b = ev.kendall_tau(emb)
        again = ev.kendall_tau(emb)
        calls = list(lib.calls)
    with np.errstate(all="ignore"):
        m = 1 - np.corrcoef(emb.numpy().astype(np.float64))
    iu = np.triu_indices(N, 1)
    x, y = m[iu], ref[iu]
    assert tau_b == float(kendalltau(x, y).statistic) and (tau_a, tau_b) == again
    assert tau_a == float(kendall_counts(x, y)[0]) / float(len(x) * (len(x) - 1) // 2)
    # the reference is sorted once and kept
    assert calls.count("hba_rank_order_f64") == 1 and calls.count("hba_kendall_tau_f64") == 2
    with emulated_device():
        with pytest.raises(ValueError):
            ev.kendall_tau(emb[:-1])


def test_kernel_launch_count():
    from hba import ops
    assert ops.kendall_kernels(1128) == 1 and ops.kendall_kernels(2048) == 1
    assert ops.kendall_kernels(4096) == 13 and ops.kendall_kernels(4097) == 14
    assert ops.kendall_kernels(1854 * 1853 // 2) == 13 + 9


def test_rsa_over_checkpoints_csv(tmp_path):
    """Without kendall the CSV is byte for byte what RESULT_COLUMNS alone gives; with it KENDALL_COLUMNS follow, with
    the values of the evaluator's own method."""
    import pandas as pd
    from hba import rsa_scale
    from hba.rsa import RSAEvaluator
    from oracle.libhba_ref import emulated_device
    from test_gpu_kendall import _data
    N = 48
    ref, emb0 = _data(N, seed=8)
    extra = torch.from_numpy(np.random.default_rng(2).standard_normal((N, 8)).astype(np.float32))

    class _Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.m = torch.nn.Parameter(torch.zeros(1))

    embed = lambda model, loaders, device: emb0 + extra * float(model.m.detach()[0])
    root = str(tmp_path)
    for run, epochs in (("base/dora", (1, 3)), ("sweep/c1/dora", (2,))):
        os.makedirs(os.path.join(root, run), exist_ok=True)
        for e in epochs:
            torch.save({"m": torch.tensor([0.5 * e])}, os.path.join(root, run, f"epoch{e}_dora_params.pth"))
    files = rsa_scale.find_dora_checkpoints(root)
    with emulated_device():
        ev = RSAEvaluator(ref, "cpu")
        plain, tau = tmp_path / "plain.csv", tmp_path / "tau.csv"
        rows, _ = rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, "cpu", output_csv=str(plain), log=None,
                                                      root=root, evaluator=ev, embed_fn=embed)
        trows, _ = rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, "cpu", output_csv=str(tau), log=None,
                                                       root=root, evaluator=ev, embed_fn=embed, kendall=True)
        m = _Model()
        m.m.data.fill_(0.5)
        want = ev.kendall_tau(embed(m, [], "cpu"))
    legacy = tmp_path / "legacy.csv"
    pd.DataFrame([{k: r[k] for k in rsa_scale.RESULT_COLUMNS} for r in rows],
                 columns=list(rsa_scale.RESULT_COLUMNS)).to_csv(legacy, index=False)
    assert plain.read_bytes() == legacy.read_bytes()
    df = pd.read_csv(tau, float_precision="round_trip")
    assert list(df.columns) == list(rsa_scale.RESULT_COLUMNS + rsa_scale.KENDALL_COLUMNS)
    row = df[df["checkpoint"] == "base/dora/epoch1_dora_params.pth"].iloc[0]
    assert (row["behavioral_rsa_tau_a"], row["behavioral_rsa_tau_b"]) == want
    assert [r["behavioral_rsa_rho"] for r in rows] == [r["behavioral_rsa_rho"] for r in trows]


def test_tool_exposes_the_kendall_flag():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "clip_rsa_over_checkpoints.py"), "--help"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "--kendall" in out.stdout


def test_gpu_test_file_dry_runs_on_the_cpu_restatement():
    """tests/test_gpu_kendall.py itself, run by pytest on the CPU with libhba served by its restatement."""
    tool = os.path.join(ROOT, "tests", "emulate_clip_gpu_tests.py")
    out = subprocess.run([sys.executable, tool, os.path.join(ROOT, "tests", "test_gpu_kendall.py")],
                         capture_output=True, text=True, timeout=1200, env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    tail = [l for l in out.stdout.splitlines() if " passed" in l][-1]
    assert "failed" not in tail and "error" not in tail and int(tail.split(" passed")[0].split()[-1]) >= 30, tail
