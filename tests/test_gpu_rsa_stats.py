"""The RSA resampling statistics on the B200 (hba_rank_order_f64, hba_rsa_perm_null, hba_rsa_bootstrap through
hba.rsa.RSAEvaluator) against a brute-force numpy / scipy oracle that builds every permuted or resampled sub-RDM
explicitly, drops the pairs of a stimulus with itself and calls scipy.stats.spearmanr: every replicate within 1e-12,
p-values and intervals equal, outputs bit-identical run to run."""
import os

import numpy as np
import pytest
import torch
from scipy.stats import spearmanr

import rsa_stats_ref  # noqa: F401  (lets tests/emulate_clip_gpu_tests.py dry-run this file on the CPU restatement)

pytestmark = pytest.mark.gpu

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _sym(r):
    """The RDM the library sees: its upper triangle, mirrored."""
    u = np.triu(np.asarray(r, dtype=np.float64), 1)
    return u + u.T


def _data(N, Dm=8, seed=0, ties=False):
    rng = np.random.default_rng(seed)
    if ties:   # few distinct rows: thousands of exactly equal RDM entries in both RDMs
        t = rng.integers(0, 3, size=(N, 3)) * np.array([1.0, 2.0, 4.0]) + np.array([0.0, 0.1, 0.3])
        e = (rng.integers(0, 3, size=(N, 3)) * np.array([1, 2, 4]) + np.array([0, 0.5, 0.25])).astype(np.float32)
    else:
        t = rng.standard_normal((N, Dm))
        e = rng.standard_normal((N, Dm)).astype(np.float32)
    with np.errstate(all="ignore"):
        ref = 1 - np.corrcoef(t)
    np.fill_diagonal(ref, 0)
    return ref, torch.from_numpy(e)


def _model_rdm(emb):
    """The model RDM exactly as the library computes it (hba_rdm_f64)."""
    from hba import ops
    N = emb.shape[0]
    rdm = torch.empty(N, N, dtype=torch.float64, device=DEV)
    ops.rdm_f64(emb.to(DEV).contiguous(), rdm, torch.empty(N * (N - 1) // 2, dtype=torch.float64, device=DEV))
    return _sym(rdm.cpu().numpy())


def _spearman(a, b):
    with np.errstate(all="ignore"):
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return float(spearmanr(a, b)[0])


def brute_perm(ref, m, N, n_perm, seed):
    rng = np.random.default_rng(seed)
    iu = np.triu_indices(N, 1)
    return np.array([_spearman(ref[iu], m[np.ix_(pi, pi)][iu]) for pi in (rng.permutation(N) for _ in range(n_perm))])


def brute_boot(ref, m, N, n_boot, seed):
    rng = np.random.default_rng(seed)
    I, J = np.triu_indices(N, 1)
    out = []
    for _ in range(n_boot):
        idx = rng.integers(0, N, size=N)
        a, b = idx[I], idx[J]
        keep = a != b
        out.append(_spearman(ref[a[keep], b[keep]], m[a[keep], b[keep]]))
    return np.array(out)


def _close(got, want, tol=1e-12):
    got, want = np.asarray(got), np.asarray(want)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = ~np.isnan(want)
    assert np.abs(got[ok] - want[ok]).max(initial=0.0) <= tol, np.abs(got[ok] - want[ok]).max()


@pytest.mark.parametrize("N,n_perm,n_boot", [(48, 300, 200), (300, 64, 48), (1854, 24, 12)])
def test_permutations_and_bootstrap_match_the_brute_force_oracle(N, n_perm, n_boot):
    from hba.rsa import RSAEvaluator, percentile_interval, permutation_pvalue
    ref, emb = _data(N, seed=N)
    ev = RSAEvaluator(ref, DEV)
    m, R = _model_rdm(emb), _sym(ref)
    rho, p, null = ev.permutation_test(emb, n_perm=n_perm, seed=7)
    want = brute_perm(R, m, N, n_perm, 7)
    _close(null, want)
    assert p == permutation_pvalue(rho, want)
    (lo, hi), reps, valid = ev.bootstrap(emb, n_boot=n_boot, seed=11, alpha=0.1)
    want = brute_boot(R, m, N, n_boot, 11)
    _close(reps, want)
    assert valid == np.isfinite(want).sum()
    wlo, whi = percentile_interval(want, 0.1)
    assert abs(lo - wlo) <= 1e-12 and abs(hi - whi) <= 1e-12
    if N <= 300:   # paired difference on identical resamples
        _, emb2 = _data(N, seed=N + 1)
        (dlo, dhi), d, _ = ev.bootstrap(emb, n_boot=n_boot, seed=11, paired_with=emb2)
        _close(d, want - brute_boot(R, _model_rdm(emb2), N, n_boot, 11))


def test_exact_ties_and_nan_rows_at_1854():
    from hba import ops
    from hba.rsa import RSAEvaluator
    N = 1854
    ref, emb = _data(N, seed=3, ties=True)
    ev = RSAEvaluator(ref, DEV)
    m, R = _model_rdm(emb), _sym(ref)
    iu = np.triu_indices(N, 1)
    assert len(np.unique(m[iu])) < 1000 and len(np.unique(R[iu])) < 1000   # thousands of exact ties
    _close(ev.permutation_test(emb, n_perm=16, seed=2)[2], brute_perm(R, m, N, 16, 2))
    _close(ev.bootstrap(emb, n_boot=12, seed=5)[1], brute_boot(R, m, N, 12, 5))
    # a NaN row and a constant row: the observed rho is NaN -> NaN p and interval
    for bad in ("nan", "const"):
        e = emb.clone()
        e[17] = float("nan") if bad == "nan" else 1.0
        rho, p, null = ev.permutation_test(e, n_perm=4)
        assert rho != rho and p != p and np.isnan(null).all()
        (lo, hi), reps, valid = ev.bootstrap(e, n_boot=4)
        assert lo != lo and hi != hi and valid == 0
    # the kernels themselves with a NaN row: exactly the resamples that draw stimulus 17 are NaN
    e = emb.clone()
    e[17] = float("nan")
    me = _model_rdm(e)
    tri = torch.from_numpy(np.ascontiguousarray(me[iu])).to(DEV)
    order = torch.empty(len(iu[0]), dtype=torch.int32, device=DEV)
    ranks = torch.empty(len(iu[0]), dtype=torch.float64, device=DEV)
    ops.rank_order_f64(tri, order, ranks, ev.rank_ws)
    ref_tri = torch.from_numpy(np.ascontiguousarray(R[iu])).to(DEV)
    ref_order = torch.empty_like(order)
    ops.rank_order_f64(ref_tri, ref_order, torch.empty_like(ranks), ev.rank_ws)
    rng = np.random.default_rng(9)
    counts = np.stack([np.bincount(rng.integers(0, N, N), minlength=N) for _ in range(12)]).astype(np.int32)
    counts[0, 17], counts[0, 18] = 0, counts[0, 18] + counts[0, 17]          # one resample without stimulus 17
    out = torch.full((12,), float("nan"), dtype=torch.float64, device=DEV)
    ws = torch.empty(ops.rsa_boot_workspace_bytes(N, 12), dtype=torch.uint8, device=DEV)
    ops.rsa_bootstrap(ref_tri, ref_order, tri, order, torch.from_numpy(counts).to(DEV), out, ws)
    got = out.cpu().numpy()
    want = []
    I, J = iu
    for c in counts:
        idx = np.repeat(np.arange(N), c)
        a, b = idx[np.triu_indices(N, 1)[0]], idx[np.triu_indices(N, 1)[1]]
        keep = a != b
        want.append(_spearman(R[a[keep], b[keep]], me[a[keep], b[keep]]))
    _close(got, np.array(want))
    assert not np.isnan(got[0]) and np.isnan(got[1:]).sum() == (counts[1:, 17] > 0).sum()


def test_outputs_are_bit_identical_run_to_run():
    from hba.rsa import RSAEvaluator
    ref, emb = _data(1854, seed=4)
    ev = RSAEvaluator(ref, DEV)
    a = ev.permutation_test(emb, n_perm=64, seed=1)[2], ev.bootstrap(emb, n_boot=24, seed=1)[1]
    b = ev.permutation_test(emb, n_perm=64, seed=1)[2], ev.bootstrap(emb, n_boot=24, seed=1)[1]
    assert all(x.tobytes() == y.tobytes() for x, y in zip(a, b))


def test_small_and_degenerate_resamples():
    """Fewer than 3 distinct stimuli in a resample, counts that do not sum to N, a permutation entry out of range:
    NaN for that replicate, the others unaffected."""
    from hba import ops
    from hba.rsa import RSAEvaluator
    N = 48
    ref, emb = _data(N, seed=6)
    ev = RSAEvaluator(ref, DEV)
    tri, order, ranks = ev._model_arrays(emb)
    ref_order = torch.empty_like(order)
    ops.rank_order_f64(ev.ref_tri, ref_order, torch.empty_like(ranks), ev.rank_ws)
    counts = np.ones((4, N), np.int32)
    counts[1] = 0
    counts[1, [3, 9]] = [20, 28]            # 2 distinct stimuli: one distinct pair, constant triangle
    counts[2, 0] = 2                        # sums to N + 1
    counts[3] = 0
    counts[3, [1, 2, 5]] = [16, 16, 16]     # 3 distinct stimuli
    out = torch.full((4,), float("nan"), dtype=torch.float64, device=DEV)
    ws = torch.empty(ops.rsa_boot_workspace_bytes(N, 4), dtype=torch.uint8, device=DEV)
    ops.rsa_bootstrap(ev.ref_tri, ref_order, tri, order, torch.from_numpy(counts).to(DEV), out, ws)
    got = out.cpu().numpy()
    assert np.isfinite(got[0]) and np.isnan(got[1]) and np.isnan(got[2]) and np.isfinite(got[3])
    assert abs(got[0] - ev(emb, want_rdm=False)[0]) <= 1e-12     # all counts 1: the plain rho
    perms = np.stack([np.arange(N), np.arange(N)]).astype(np.int32)
    perms[1, 5] = N
    out = torch.full((2,), float("nan"), dtype=torch.float64, device=DEV)
    ws = torch.empty(ops.rsa_perm_workspace_bytes(N, 2), dtype=torch.uint8, device=DEV)
    ops.rsa_perm_null(ev.ref_ranks, ranks, torch.from_numpy(perms).to(DEV), out, ws)
    got = out.cpu().numpy()
    assert abs(got[0] - ev(emb, want_rdm=False)[0]) <= 1e-12 and np.isnan(got[1])


def test_argument_errors_are_reported_not_faults():
    from hba import _lib
    lib = _lib.load()
    N, P = 48, 48 * 47 // 2
    x = torch.zeros(P, dtype=torch.float64, device=DEV)
    o = torch.zeros(P, dtype=torch.int32, device=DEV)
    perms = torch.zeros(4, N, dtype=torch.int32, device=DEV)
    rho = torch.zeros(4, dtype=torch.float64, device=DEV)
    ws = torch.zeros(lib.hba_rsa_boot_workspace_bytes(N, 4), dtype=torch.uint8, device=DEV)
    p = lambda t: t.data_ptr()
    cases = [
        (lambda: lib.hba_rsa_perm_null(p(x), p(x), 2, p(perms), 4, p(rho), p(ws), ws.numel(), None), "N=2"),
        (lambda: lib.hba_rsa_perm_null(p(x), p(x), 3000, p(perms), 4, p(rho), p(ws), ws.numel(), None), "N=3000"),
        (lambda: lib.hba_rsa_perm_null(p(x), p(x), N, p(perms), 0, p(rho), p(ws), ws.numel(), None), "n_perm=0"),
        (lambda: lib.hba_rsa_perm_null(p(x), None, N, p(perms), 4, p(rho), p(ws), ws.numel(), None), "null pointer"),
        (lambda: lib.hba_rsa_perm_null(p(x), p(x), N, p(perms), 4, p(rho), p(ws), 16, None), "workspace"),
        (lambda: lib.hba_rsa_perm_null(p(x), p(x), N, p(perms) + 2, 4, p(rho), p(ws), ws.numel(), None), "misaligned"),
        (lambda: lib.hba_rsa_bootstrap(p(x), p(o), p(x), p(o), None, None, N, p(perms), 0, p(rho), None, p(ws), ws.numel(),
                               None), "n_boot=0"),
        (lambda: lib.hba_rsa_bootstrap(p(x), p(o), p(x), p(o), p(x), None, N, p(perms), 4, p(rho), None, p(ws), ws.numel(),
                               None), "together"),
        (lambda: lib.hba_rsa_bootstrap(p(x), p(o), p(x), p(o), None, None, N, p(perms), 4, p(rho), None, p(ws), 16, None),
         "workspace"),
        (lambda: lib.hba_rsa_bootstrap(p(x), p(o), p(x), p(o), None, None, 2300, p(perms), 4, p(rho), None, p(ws),
                               ws.numel(), None), "N=2300"),
        (lambda: lib.hba_rank_order_f64(p(x), 0, p(o), p(x), p(ws), ws.numel(), None), "bad arguments"),
    ]
    for call, what in cases:
        assert call() == -22, what
        assert what in _lib.last_error() or what.startswith(("null", "together", "bad")), (what, _lib.last_error())
    torch.cuda.synchronize()


def test_rsa_over_checkpoints_writes_the_new_columns(tmp_path):
    """hba.rsa_scale end to end on the device evaluator: the default columns without the flags, the statistics
    columns with them, the same rho either way; the statistics equal the evaluator's."""
    import pandas as pd
    from hba import rsa_scale
    from hba.rsa import RSAEvaluator
    N = 48
    ref, emb0 = _data(N, seed=12)
    for e in (1, 2):
        os.makedirs(tmp_path / "run" / "dora", exist_ok=True)
        torch.save({"m": torch.tensor([1.0 + e])}, tmp_path / "run" / "dora" / f"epoch{e}_dora_params.pth")

    class _Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.m = torch.nn.Parameter(torch.zeros(1))

    extra = torch.from_numpy(np.random.default_rng(1).standard_normal((N, 8)).astype(np.float32))
    embed = lambda model, loaders, device: (emb0 + extra * float(model.m.detach()[0])).to(device)
    files = rsa_scale.find_dora_checkpoints(str(tmp_path))
    ev = RSAEvaluator(ref, DEV)
    out = {}
    for flags in ((0, 0), (200, 50)):
        csv = tmp_path / f"rsa_{flags[0]}.csv"
        rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, DEV, output_csv=str(csv), log=None,
                                            root=str(tmp_path), evaluator=ev, embed_fn=embed, n_perm=flags[0],
                                            n_boot=flags[1], seed=3)
        out[flags] = pd.read_csv(csv, float_precision="round_trip")
    plain, stats = out[(0, 0)], out[(200, 50)]
    assert list(plain.columns) == list(rsa_scale.RESULT_COLUMNS)
    assert list(stats.columns) == list(rsa_scale.RESULT_COLUMNS + rsa_scale.PERMUTATION_COLUMNS
                                       + rsa_scale.BOOTSTRAP_COLUMNS)
    assert (plain["behavioral_rsa_rho"] == stats["behavioral_rsa_rho"]).all()
    m = _Model()
    m.m.data.fill_(2.0)
    e = embed(m, [], DEV)
    assert stats["behavioral_rsa_p_perm"][0] == ev.permutation_test(e, n_perm=200, seed=3)[1]
    (lo, hi), _, valid = ev.bootstrap(e, n_boot=50, seed=3)
    assert (stats["behavioral_rsa_ci_low"][0], stats["behavioral_rsa_ci_high"][0]) == (lo, hi)
    assert stats["behavioral_rsa_boot_valid"][0] == valid == 50
