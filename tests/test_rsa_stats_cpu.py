"""RSA resampling statistics (hba.rsa.RSAEvaluator.permutation_test / .bootstrap) on the CPU: the weighted-rank identity
the bootstrap kernels rest on, the host API on the CPU restatement of libhba against a brute-force numpy / scipy
oracle, the seeds, the p-value and interval formulas, the CSV of hba.rsa_scale, and a dry run of the GPU test file."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy.stats import rankdata

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import rsa_stats_ref  # noqa: E402,F401  (the CPU restatement of the resampling entries, served by emulated_device)
from test_gpu_rsa_stats import _data, _sym, brute_boot, brute_perm  # noqa: E402  (the oracle the GPU tests use)


def _rdm(emb):
    with np.errstate(all="ignore"):
        r = 1 - np.corrcoef(np.asarray(emb, dtype=np.float64))
    np.fill_diagonal(r, 0)
    return _sym(r)


@pytest.mark.parametrize("seed", range(6))
def test_weighted_ranks_equal_rankdata_of_the_expanded_multiset(seed):
    """S_g + (W_g + 1) / 2 over the fixed sorted order = rankdata(..., 'average') of the values repeated w times,
    with forced ties (values from a small set, -0.0 and +0.0 equal) and with NaN entries of weight 0."""
    from rsa_stats_ref import sorted_order, weighted_average_ranks
    rng = np.random.default_rng(seed)
    n = 300
    x = rng.integers(0, 12, n).astype(np.float64) / 4 - 1.0
    x[rng.integers(0, n, 10)] = -0.0
    x[rng.integers(0, n, 10)] = 0.0
    w = rng.integers(0, 4, n)
    if seed % 2:
        nan_at = rng.choice(n, 7, replace=False)
        x[nan_at[:4]] = np.nan
        x[nan_at[4:]] = -np.nan
        w[nan_at] = 0
    order = sorted_order(x)[0]
    r = weighted_average_ranks(x, order, w)
    live = w > 0
    expanded = np.repeat(x[live], w[live])
    want = rankdata(expanded, method="average")
    assert np.array_equal(np.repeat(r[live], w[live]), want[np.argsort(np.repeat(np.flatnonzero(live), w[live]),
                                                                       kind="stable")])
    # and with a NaN of weight > 0 scipy propagates: the replicate is NaN
    if seed % 2:
        assert np.isnan(rankdata(np.append(expanded, np.nan), nan_policy="propagate")).all()


def test_weighted_ranks_with_all_weights_one_are_rankdata():
    from rsa_stats_ref import sorted_order, weighted_average_ranks
    x = np.random.default_rng(0).integers(0, 5, 200).astype(np.float64)
    assert np.array_equal(weighted_average_ranks(x, sorted_order(x)[0], np.ones(200, np.int64)), rankdata(x))


@pytest.mark.parametrize("N", [48, 120])
def test_host_api_matches_the_brute_force_oracle(N):
    from hba.rsa import RSAEvaluator, percentile_interval, permutation_pvalue
    from oracle.libhba_ref import emulated_device
    ref, emb = _data(N, seed=N)
    _, emb2 = _data(N, seed=N + 1)
    with emulated_device():
        ev = RSAEvaluator(ref, "cpu")
        rho, p, null = ev.permutation_test(emb, n_perm=60, seed=4)
        (lo, hi), reps, valid = ev.bootstrap(emb, n_boot=40, seed=5)
        (dlo, dhi), d, dvalid = ev.bootstrap(emb, n_boot=40, seed=5, paired_with=emb2)
    R, m, m2 = _sym(ref), _rdm(emb), _rdm(emb2)
    want = brute_perm(R, m, N, 60, 4)
    assert np.abs(null - want).max() <= 1e-12 and p == permutation_pvalue(rho, want)
    want = brute_boot(R, m, N, 40, 5)
    assert np.abs(reps - want).max() <= 1e-12 and valid == 40
    assert np.allclose((lo, hi), percentile_interval(want), rtol=0, atol=1e-12)
    want_d = want - brute_boot(R, m2, N, 40, 5)
    assert np.abs(d - want_d).max() <= 1e-12 and dvalid == 40
    assert np.allclose((dlo, dhi), percentile_interval(want_d), rtol=0, atol=1e-12)


def test_seeds_reproduce_and_differ():
    from hba.rsa import RSAEvaluator
    from oracle.libhba_ref import emulated_device
    ref, emb = _data(48, seed=1)
    with emulated_device():
        ev = RSAEvaluator(ref, "cpu")
        a = ev.permutation_test(emb, n_perm=30, seed=3)[2], ev.bootstrap(emb, n_boot=20, seed=3)[1]
        b = ev.permutation_test(emb, n_perm=30, seed=3)[2], ev.bootstrap(emb, n_boot=20, seed=3)[1]
        c = ev.permutation_test(emb, n_perm=30, seed=4)[2], ev.bootstrap(emb, n_boot=20, seed=4)[1]
        # chunking does not change the draws
        import hba.rsa as rsa
        saved = rsa.STATS_CHUNK_BYTES
        try:
            rsa.STATS_CHUNK_BYTES = 1
            d = ev.permutation_test(emb, n_perm=30, seed=3)[2], ev.bootstrap(emb, n_boot=20, seed=3)[1]
        finally:
            rsa.STATS_CHUNK_BYTES = saved
    assert all(np.array_equal(x, y) for x, y in zip(a, b)) and all(np.array_equal(x, y) for x, y in zip(a, d))
    assert not any(np.array_equal(x, y) for x, y in zip(a, c))


def test_pvalue_and_interval_formulas():
    from hba.rsa import check_permutations, percentile_interval, permutation_pvalue
    null = np.array([0.1, 0.3, np.nan, 0.2, 0.5])
    assert permutation_pvalue(0.3, null) == (1 + 2) / 6
    assert permutation_pvalue(0.9, null) == 1 / 6
    assert np.isnan(permutation_pvalue(float("nan"), null))
    reps = np.array([np.nan, 1.0, 2.0, 3.0, 4.0, np.nan, 5.0])
    assert percentile_interval(reps, 0.5) == tuple(np.quantile([1.0, 2, 3, 4, 5], [0.25, 0.75]))
    assert all(np.isnan(percentile_interval(np.full(3, np.nan))))
    check_permutations(np.array([[2, 0, 1], [0, 1, 2]]), 3)
    with pytest.raises(ValueError):
        check_permutations(np.array([[2, 2, 1]]), 3)


def test_nan_observed_rho_gives_nan_statistics():
    from hba.rsa import RSAEvaluator
    from oracle.libhba_ref import emulated_device
    ref, emb = _data(48, seed=2)
    emb[5] = 1.0                       # constant row: its correlations are NaN
    with emulated_device():
        ev = RSAEvaluator(ref, "cpu")
        rho, p, null = ev.permutation_test(emb, n_perm=5)
        (lo, hi), reps, valid = ev.bootstrap(emb, n_boot=5)
    assert rho != rho and p != p and np.isnan(null).all() and lo != lo and hi != hi and valid == 0


def _write_checkpoints(root, N):
    for run, epochs in (("base/dora", (1, 3)), ("sweep/c1/dora", (2,))):
        os.makedirs(os.path.join(root, run), exist_ok=True)
        for e in epochs:
            torch.save({"m": torch.tensor([0.5 * e])}, os.path.join(root, run, f"epoch{e}_dora_params.pth"))


def test_rsa_over_checkpoints_csv(tmp_path):
    """With n_perm = n_boot = 0 the CSV is byte for byte what RESULT_COLUMNS alone gives; with them the statistics
    columns follow, with the values of the evaluator's own methods."""
    import pandas as pd
    from hba import rsa_scale
    from hba.rsa import RSAEvaluator
    from oracle.libhba_ref import emulated_device
    N = 48
    ref, emb0 = _data(N, seed=8)
    extra = torch.from_numpy(np.random.default_rng(2).standard_normal((N, 8)).astype(np.float32))

    class _Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.m = torch.nn.Parameter(torch.zeros(1))

    embed = lambda model, loaders, device: emb0 + extra * float(model.m.detach()[0])
    root = str(tmp_path)
    _write_checkpoints(root, N)
    files = rsa_scale.find_dora_checkpoints(root)
    with emulated_device():
        ev = RSAEvaluator(ref, "cpu")
        plain = tmp_path / "plain.csv"
        rows, _ = rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, "cpu", output_csv=str(plain), log=None,
                                                      root=root, evaluator=ev, embed_fn=embed)
        stats = tmp_path / "stats.csv"
        srows, _ = rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, "cpu", output_csv=str(stats),
                                                       log=None, root=root, evaluator=ev, embed_fn=embed, n_perm=40,
                                                       n_boot=30, seed=1)
        m = _Model()
        m.m.data.fill_(0.5)
        e1 = embed(m, [], "cpu")
        p1 = ev.permutation_test(e1, n_perm=40, seed=1)[1]
        (lo, hi), _, valid = ev.bootstrap(e1, n_boot=30, seed=1)
    legacy = tmp_path / "legacy.csv"
    pd.DataFrame([{k: r[k] for k in rsa_scale.RESULT_COLUMNS} for r in rows],
                 columns=list(rsa_scale.RESULT_COLUMNS)).to_csv(legacy, index=False)
    assert plain.read_bytes() == legacy.read_bytes()
    df = pd.read_csv(stats, float_precision="round_trip")
    assert list(df.columns) == list(rsa_scale.RESULT_COLUMNS + rsa_scale.PERMUTATION_COLUMNS
                                    + rsa_scale.BOOTSTRAP_COLUMNS)
    assert list(df["checkpoint"]) == [os.path.relpath(f, root) for f in sorted(files)]
    row = df[df["checkpoint"] == "base/dora/epoch1_dora_params.pth"].iloc[0]
    assert row["behavioral_rsa_p_perm"] == p1 and (row["behavioral_rsa_ci_low"], row["behavioral_rsa_ci_high"]) == (lo, hi)
    assert row["behavioral_rsa_boot_valid"] == valid == 30
    assert [r["behavioral_rsa_rho"] for r in rows] == [r["behavioral_rsa_rho"] for r in srows]


def test_tool_exposes_the_statistics_flags():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "clip_rsa_over_checkpoints.py"), "--help"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and all(f in out.stdout for f in ("--permutations", "--bootstrap", "--seed"))


def test_gpu_test_file_dry_runs_on_the_cpu_restatement():
    """tests/test_gpu_rsa_stats.py itself, run by pytest on the CPU with libhba served by its restatement."""
    tool = os.path.join(ROOT, "tests", "emulate_clip_gpu_tests.py")
    out = subprocess.run([sys.executable, tool, os.path.join(ROOT, "tests", "test_gpu_rsa_stats.py")],
                         capture_output=True, text=True, timeout=1200, env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    tail = [l for l in out.stdout.splitlines() if " passed" in l][-1]
    assert "failed" not in tail and "error" not in tail and int(tail.split(" passed")[0].split()[-1]) >= 8, tail
