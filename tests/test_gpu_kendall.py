"""Kendall's tau on the B200 (hba_kendall_tau_f64 through hba.ops and hba.rsa.RSAEvaluator.kendall_tau) against the
exact numpy oracle of tests/kendall_ref.py: the four pair counts equal, tau_b == scipy.stats.kendalltau, tau_a == S/n0,
at the RSA sizes and at sizes on both sides of every size threshold of the kernels (one CTA up to n = 2048, tiles of
4096, one merge level per doubling beyond)."""
import os
import warnings

import numpy as np
import pytest
import torch
from scipy.stats import kendalltau

from kendall_ref import kendall_counts  # (also lets tests/emulate_clip_gpu_tests.py dry-run this file on the CPU)

pytestmark = pytest.mark.gpu

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _scipy_tau_b(x, y):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return float(kendalltau(x, y).statistic)


def _data(N, Dm=8, seed=0):
    rng = np.random.default_rng(seed)
    with np.errstate(all="ignore"):
        ref = 1 - np.corrcoef(rng.standard_normal((N, Dm)))
    np.fill_diagonal(ref, 0)
    return ref, torch.from_numpy(rng.standard_normal((N, Dm)).astype(np.float32))


def _model_tri(emb):
    """The model triangle exactly as the library computes it (hba_rdm_f64)."""
    from hba import ops
    N = emb.shape[0]
    tri = torch.empty(N * (N - 1) // 2, dtype=torch.float64, device=DEV)
    ops.rdm_f64(emb.to(DEV).contiguous(), None, tri)
    return tri.cpu().numpy()


def _kendall(x, y):
    """(counts, (tau_a, tau_b)) of the library for host vectors x, y; y sorted by hba_rank_order_f64."""
    from hba import ops
    n = len(x)
    xd = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(DEV)
    yd = torch.from_numpy(np.ascontiguousarray(y, dtype=np.float64)).to(DEV)
    order = torch.empty(n, dtype=torch.int32, device=DEV)
    rank_ws = torch.empty(max(ops.rank_workspace_bytes(n), 256), dtype=torch.uint8, device=DEV)
    ops.rank_order_f64(yd, order, torch.empty(n, dtype=torch.float64, device=DEV), rank_ws)
    counts = torch.empty(4, dtype=torch.int64, device=DEV)
    tau = torch.empty(2, dtype=torch.float64, device=DEV)
    ws = torch.empty(ops.kendall_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    ops.kendall_tau_f64(xd, yd, order, counts, tau, ws)
    return tuple(counts.cpu().tolist()), tuple(tau.cpu().tolist())


def _check(x, y, counts, taus):
    n = len(x)
    want = kendall_counts(x, y)
    assert counts == want, (n, counts, want)
    tau_b = _scipy_tau_b(x, y)
    assert taus[1] == tau_b or (taus[1] != taus[1] and tau_b != tau_b), (n, taus[1], tau_b)
    if tau_b == tau_b:
        assert taus[0] == float(want[0]) / float(n * (n - 1) // 2)
    else:   # a constant side
        assert taus[0] != taus[0] and n * (n - 1) // 2 in want[1:3]


@pytest.mark.parametrize("n", [2, 3, 1128, 2048, 2049, 4096, 4097, 8192, 8193, 16385, 100003])
@pytest.mark.parametrize("kind", ["continuous", "ties"])
def test_counts_at_every_size_threshold(n, kind):
    """Both sides of the one-CTA bound (2048), of one tile (4096) and of the first merge levels (8192, 16384)."""
    rng = np.random.default_rng(n)
    if kind == "continuous":
        x, y = rng.standard_normal(n), rng.standard_normal(n)
        y[: n // 3] = x[: n // 3]   # some association
    else:   # large tie groups in both, -0.0 and +0.0 equal
        x = rng.integers(-3, 4, n).astype(np.float64) * 0.5
        y = rng.integers(0, 5, n).astype(np.float64) + (x > 0)
        x[x == 0] = np.where(rng.random((x == 0).sum()) < 0.5, -0.0, 0.0)
    counts, taus = _kendall(x, y)
    _check(x, y, counts, taus)


@pytest.mark.parametrize("N", [48, 300, 1854])
def test_rdms_against_the_oracle_and_scipy(N):
    from hba.rsa import RSAEvaluator
    ref, emb = _data(N, seed=N)
    ev = RSAEvaluator(ref, DEV)
    tau_a, tau_b = ev.kendall_tau(emb)
    x, y = _model_tri(emb), ref[np.triu_indices(N, 1)]
    S = kendall_counts(x, y)[0]
    assert tau_b == _scipy_tau_b(x, y) and tau_a == float(S) / float(len(x) * (len(x) - 1) // 2)


def test_categorical_reference_and_quantised_embeddings_at_1854():
    """A same/different-category reference (two distinct values) and embeddings with large tie groups in x."""
    from hba.rsa import RSAEvaluator
    N = 1854
    rng = np.random.default_rng(5)
    cat = rng.integers(0, 27, N)
    ref = (cat[:, None] != cat[None, :]).astype(np.float64)
    kind = np.where(rng.random(N) < 0.7, cat % 16, rng.integers(0, 16, N))   # 16 distinct rows, mostly by category
    bits = (kind[:, None] >> np.arange(4)) & 1
    emb = torch.from_numpy((bits * np.array([1.0, 2.0, 4.0, 8.0]) + 0.37 * np.arange(4)).astype(np.float32))
    ev = RSAEvaluator(ref, DEV)
    x, y = _model_tri(emb), ref[np.triu_indices(N, 1)]
    assert len(np.unique(x)) < 1000 and len(np.unique(y)) == 2
    _check(x, y, *_kendall(x, y))
    tau_a, tau_b = ev.kendall_tau(emb)
    assert tau_b == _scipy_tau_b(x, y) and abs(tau_a) < abs(tau_b)   # tau-a does not reward predicted ties


@pytest.mark.parametrize("N", [48, 1854])
def test_nan_and_constant_inputs(N):
    from hba.rsa import RSAEvaluator
    ref, emb = _data(N, seed=2)
    ev = RSAEvaluator(ref, DEV)
    e = emb.clone()
    e[17] = float("nan")
    x, y = _model_tri(e), ref[np.triu_indices(N, 1)]
    counts, taus = _kendall(x, y)
    assert counts == (-1, -1, -1, -1) and all(t != t for t in taus)
    assert all(t != t for t in ev.kendall_tau(e))
    # constant embeddings: every correlation is NaN, so is every RDM entry
    assert all(t != t for t in ev.kendall_tau(torch.ones_like(emb)))
    # a constant model triangle and a constant reference: the counts are written, the taus are NaN
    x = _model_tri(emb)
    for xx, yy in ((np.full_like(x, 0.25), y), (x, np.full_like(y, 0.5))):
        counts, taus = _kendall(xx, yy)
        assert counts == kendall_counts(xx, yy) and all(t != t for t in taus)
        assert np.isnan(_scipy_tau_b(xx, yy))
    const_ref = np.full((N, N), 0.5)
    np.fill_diagonal(const_ref, 0)
    assert all(t != t for t in RSAEvaluator(const_ref, DEV).kendall_tau(emb))


def test_reruns_are_bit_identical():
    from hba.rsa import RSAEvaluator
    ref, emb = _data(1854, seed=4)
    ev = RSAEvaluator(ref, DEV)
    a = [ev.kendall_tau(emb) for _ in range(3)]
    assert all(np.array(t).tobytes() == np.array(a[0]).tobytes() for t in a)


@pytest.mark.parametrize("n", [1128, 100003])
def test_captured_graph_replay_equals_eager(n):
    from hba import ops
    rng = np.random.default_rng(9)
    x = torch.from_numpy(rng.integers(0, 50, n).astype(np.float64)).to(DEV)
    y = torch.from_numpy(rng.standard_normal(n)).to(DEV)
    order = torch.empty(n, dtype=torch.int32, device=DEV)
    rank_ws = torch.empty(max(ops.rank_workspace_bytes(n), 256), dtype=torch.uint8, device=DEV)
    ops.rank_order_f64(y, order, torch.empty(n, dtype=torch.float64, device=DEV), rank_ws)
    ws = torch.empty(ops.kendall_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    eager_c, eager_t = torch.empty(4, dtype=torch.int64, device=DEV), torch.empty(2, dtype=torch.float64, device=DEV)
    ops.kendall_tau_f64(x, y, order, eager_c, eager_t, ws)
    c = torch.full((4,), 7, dtype=torch.int64, device=DEV)
    t = torch.zeros(2, dtype=torch.float64, device=DEV)
    if torch.device(DEV).type == "cuda":
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(s), torch.cuda.graph(g, stream=s):
            ops.kendall_tau_f64(x, y, order, c, t, ws)
        torch.cuda.current_stream().wait_stream(s)
        g.replay()
        torch.cuda.synchronize()
    else:   # the CPU dry run has no graphs: call by call
        ops.kendall_tau_f64(x, y, order, c, t, ws)
    assert c.cpu().tolist() == eager_c.cpu().tolist() and t.cpu().numpy().tobytes() == eager_t.cpu().numpy().tobytes()


def test_argument_errors_are_reported_not_faults():
    from hba import _lib
    lib = _lib.load()
    n = 5000
    x = torch.zeros(n, dtype=torch.float64, device=DEV)
    o = torch.zeros(n, dtype=torch.int32, device=DEV)
    c = torch.zeros(4, dtype=torch.int64, device=DEV)
    t = torch.zeros(2, dtype=torch.float64, device=DEV)
    ws = torch.zeros(lib.hba_kendall_workspace_bytes(n), dtype=torch.uint8, device=DEV)
    p = lambda a: a.data_ptr()
    cases = [
        (lambda: lib.hba_kendall_tau_f64(p(x), p(x), p(o), 1, p(c), p(t), p(ws), ws.numel(), None), "n=1"),
        (lambda: lib.hba_kendall_tau_f64(p(x), p(x), p(o), 1 << 30, p(c), p(t), p(ws), ws.numel(), None),
         "n=1073741824"),
        (lambda: lib.hba_kendall_tau_f64(p(x), None, p(o), n, p(c), p(t), p(ws), ws.numel(), None), "null pointer"),
        (lambda: lib.hba_kendall_tau_f64(p(x), p(x), p(o), n, p(c), None, p(ws), ws.numel(), None), "null pointer"),
        (lambda: lib.hba_kendall_tau_f64(p(x) + 4, p(x), p(o), 100, p(c), p(t), p(ws), ws.numel(), None),
         "misaligned"),
        (lambda: lib.hba_kendall_tau_f64(p(x), p(x), p(o), n, p(c), p(t), p(ws), 16, None), "workspace"),
        (lambda: lib.hba_kendall_tau_f64(p(x), p(x), p(o), n, p(c), p(t), None, ws.numel(), None), "workspace"),
    ]
    for call, what in cases:
        assert call() == -22, what
        assert what in _lib.last_error(), (what, _lib.last_error())
    with pytest.raises(RuntimeError, match="workspace"):
        from hba import ops
        ops.kendall_tau_f64(x, x, o, c, t, ws[:16])
    # an order entry out of range or an order that does not sort y: counts -1, NaN, no fault
    for n_ in (100, n):
        y = torch.arange(n_, dtype=torch.float64, device=DEV)
        for bad in ("range", "unsorted"):
            order = torch.arange(n_, dtype=torch.int32, device=DEV)
            order[n_ // 2] = n_ + 5 if bad == "range" else 0
            assert lib.hba_kendall_tau_f64(p(y), p(y), p(order), n_, p(c), p(t), p(ws), ws.numel(), None) == 0
            assert c.cpu().tolist() == [-1] * 4 and torch.isnan(t).all()
    torch.cuda.synchronize()


def test_rsa_over_checkpoints_with_kendall(tmp_path):
    """hba.rsa_scale end to end on the device evaluator: the default columns without the flag, KENDALL_COLUMNS with it,
    the same rho either way, the taus equal to the evaluator's."""
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
    for kendall in (False, True):
        csv = tmp_path / f"rsa_{kendall}.csv"
        rsa_scale.clip_rsa_over_checkpoints(_Model(), [], ref, files, DEV, output_csv=str(csv), log=None,
                                            root=str(tmp_path), evaluator=ev, embed_fn=embed, kendall=kendall)
        out[kendall] = pd.read_csv(csv, float_precision="round_trip")
    assert list(out[False].columns) == list(rsa_scale.RESULT_COLUMNS)
    assert list(out[True].columns) == list(rsa_scale.RESULT_COLUMNS + rsa_scale.KENDALL_COLUMNS)
    assert (out[False]["behavioral_rsa_rho"] == out[True]["behavioral_rsa_rho"]).all()
    m = _Model()
    m.m.data.fill_(2.0)
    tau_a, tau_b = ev.kendall_tau(embed(m, [], DEV))
    assert (out[True]["behavioral_rsa_tau_a"][0], out[True]["behavioral_rsa_tau_b"][0]) == (tau_a, tau_b)
