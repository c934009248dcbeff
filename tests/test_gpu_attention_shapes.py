"""Every attention kernel of libhba at every sequence-length branch, against the fp64 reference of
tests/attention_ref.py, row by row and sequence by sequence.

Errors are per row: for each 64-element output row (one head of one token), max |got - ref| over
max |ref row|.  Tolerances: fp32 CUDA-core forward 2e-5, fp32-math backward (dQKV) 2e-4, tensor-core
forward 1e-2, bf16 backward 1.5e-2, lse 2e-3 absolute (log2 domain).  The spiked inputs put more
than 90 % of chosen rows' softmax mass on chosen keys (tile edges, the last tensor-core key, the
fp32 extra key 256, the left-over query rows), so a branch that mishandles one key or row fails.

Also: production shapes, bit-identical slicing and permutation of sequences, isolation of a sequence
from non-finite values in the next one, layout canaries (padded leading dimensions) and argument
rejection."""
import contextlib
import os

import pytest
import torch

from attention_ref import (SIMT_MAX_T, TC_BWD_MAX_T, TC_FWD_MAX_T, reference, reference_row0, row_err,
                           simt_bwd_fits, spike_pairs, spiked_qkv)

pytestmark = pytest.mark.gpu

DEV = "cuda"
SWEEP_T = [1, 2, 15, 16, 17, 31, 33, 50, 64, 65, 77, 127, 128, 129, 130, 136, 137, 144, 160, 192, 197, 203,
           204, 208, 255, 256, 257, 258, 288]
TOL_F32, TOL_F32_BWD, TOL_TC, TOL_BF16_BWD, TOL_LSE = 2e-5, 2e-4, 1e-2, 1.5e-2, 2e-3
SENTINEL = 777.0
HBA_ERR_ARG = -22
WORST = {}   # path -> worst per-row error over the module (printed at its end)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst per-row error by path:")
        for k in sorted(WORST):
            print(f"  {k:28s} {WORST[k]:.3e}")


def _ops():
    import hba  # noqa: F401
    from hba import ops
    return ops


def _record(path, e, tol):
    WORST[path] = max(WORST.get(path, 0.0), e)
    assert e < tol, (path, e, tol)


class Alloc:
    """Output buffers filled with SENTINEL; with `pad`, each is a view of a buffer with `pad` extra
    columns and one extra row, so that writes outside the logical shape can be detected."""

    def __init__(self, pad=0):
        self.pad, self.bufs = pad, []

    def __call__(self, rows, cols, dtype, pad=None):
        p = self.pad if pad is None else pad
        buf = torch.full((rows + (1 if self.pad else 0), cols + p), SENTINEL, dtype=dtype, device=DEV)
        self.bufs.append((buf, rows, cols, buf.clone()))
        return buf[:rows, :cols]

    def assert_outside_untouched(self):
        for buf, rows, cols, init in self.bufs:
            mask = torch.ones_like(buf, dtype=torch.bool)
            mask[:rows, :cols] = False
            assert torch.equal(buf[mask], init[mask]), "write outside the logical output"


@contextlib.contextmanager
def _simt(on):
    """HBA_ATTN_SIMT=1 sends bf16 hba_attention_fwd calls to the CUDA-core kernel (read on every call)."""
    old = os.environ.get("HBA_ATTN_SIMT")
    if on:
        os.environ["HBA_ATTN_SIMT"] = "1"
    try:
        yield
    finally:
        if old is None:
            os.environ.pop("HBA_ATTN_SIMT", None)
        else:
            os.environ["HBA_ATTN_SIMT"] = old


# ---------------------------------------------------------------------------------------- kernels
# Each entry: accepts(T, causal), qkv dtype, dO dtype (None: forward only; "row0": fp32 [B, H*64]),
# run(ops, qkv, do, B, T, H, causal, alloc) -> {name: output}, check(outs, qkv, do, B, T, H, causal).
def _fwd(ops, qkv, B, T, H, causal, alloc, *, out=True, f32=True, split=False, simt=False, row0=False):
    d = H * 64
    rows = B if row0 else B * T
    res, op = {}, None
    if out:
        v = alloc(rows, 2 * d if split else d, torch.bfloat16)
        op = ops.Operand(v, rows, d, d if split else 0)
        res["out"] = v
    if f32:
        res["out_f32"] = alloc(rows, d, torch.float32, pad=alloc.pad // 2)
    with _simt(simt):
        ops.attention_fwd(qkv, B, T, H, causal=causal, first_row_only=row0, out=op, out_f32=res.get("out_f32"))
    return res


def _out_value(outs, d):
    o = outs["out"]
    return o[:, :d].double() + (o[:, d:2 * d].double() if o.shape[1] > d else 0)


def _check_fwd(tol, name, split=False, row0=False):
    def check(outs, qkv, do, B, T, H, causal):
        d = H * 64
        want = (reference_row0(qkv, B, T, H) if row0 else reference(qkv, B, T, H, causal))["o"]
        if "out_f32" in outs:
            _record(name + ".out_f32", row_err(outs["out_f32"], want), tol)
        if "out" in outs:
            _record(name + (".out_hi_lo" if split else ".out"), row_err(_out_value(outs, d), want), tol)
        if T == 1:   # one key: O is V exactly (the bf16 hi/lo split of an fp32 V is not exact)
            v = qkv[:, 2 * d:3 * d].float()
            if "out_f32" in outs:   # (tensor cores: p = 2^(s*c - max*c) is 1 to within an ulp of s*c)
                torch.testing.assert_close(outs["out_f32"], v, rtol=1e-6, atol=0, msg=f"{name}: O != V at T = 1")
            if "out" in outs and not split:
                assert torch.equal(outs["out"], v.to(torch.bfloat16)), (name, "out")
        if "out" in outs and "out_f32" in outs and not split:
            assert torch.equal(outs["out"], outs["out_f32"].to(torch.bfloat16)), name
    return check


def _run_lse(ops, qkv, do, B, T, H, causal, alloc, bwd):
    d = H * 64
    out = alloc(B * T, d, torch.bfloat16)
    lse = alloc(1, B * H * T, torch.float32, pad=alloc.pad // 2)
    ops.attention_fwd_lse(qkv, B, T, H, out, lse, causal=causal)
    res = {"out": out, "lse": lse}
    if bwd:
        dq = alloc(B * T, 3 * d, torch.bfloat16)
        ops.attention_bwd_lse(qkv, B, T, H, out, do, lse, dq, causal=causal)
        res["dqkv"] = dq
    return res


def _check_lse(bwd):
    def check(outs, qkv, do, B, T, H, causal):
        r = reference(qkv, B, T, H, causal)
        _record("fwd_lse.out", row_err(outs["out"], r["o"]), TOL_TC)
        e = float((outs["lse"].double().view(B, H, T) - r["lse"]).abs().max())
        _record("fwd_lse.lse_abs", e, TOL_LSE)
        if bwd:
            # D_i = dO_i . O_i comes from the forward's bf16 O handed to the kernel
            rb = reference(qkv, B, T, H, causal, d_out=do, o_for_d=outs["out"])
            _record("bwd_lse.dqkv", row_err(outs["dqkv"], rb["dqkv"]), TOL_BF16_BWD)
    return check


def _run_row0_bwd(ops, qkv, do, B, T, H, causal, alloc):
    dq = alloc(B * T, 3 * H * 64, torch.float32, pad=alloc.pad // 2)
    ops.attention_bwd_row0(qkv, B, T, H, do, dq)
    return {"dqkv": dq}


def _check_row0_bwd(name):
    def check(outs, qkv, do, B, T, H, causal):
        _record(name, row_err(outs["dqkv"], reference_row0(qkv, B, T, H, d_out=do)["dqkv"]), TOL_F32_BWD)
    return check


def _run_bwd(ops, qkv, do, B, T, H, causal, alloc, dq_dtype):
    dq = alloc(B * T, 3 * H * 64, dq_dtype, pad=alloc.pad if dq_dtype == torch.bfloat16 else alloc.pad // 2)
    ops.attention_bwd(qkv, B, T, H, do, dq, causal=causal)
    return {"dqkv": dq}


def _check_bwd(name, tol, round_do=False):
    """round_do: the (bf16 qkv, fp32 dO) form stages dO in the same bf16 shared-memory tiles as Q, K, V, so it
    computes the gradient of bf16(dO).  Against the fp32 dO that rounding alone moves rows whose gradient
    nearly cancels (causal rows with two or three keys) by up to ~0.3 of their size."""
    def check(outs, qkv, do, B, T, H, causal):
        d_out = do.to(torch.bfloat16) if round_do else do
        _record(name, row_err(outs["dqkv"], reference(qkv, B, T, H, causal, d_out=d_out)["dqkv"]), tol)
    return check


BF, F32 = torch.bfloat16, torch.float32
KERNELS = {
    "tc.out": (lambda T, c: T <= TC_FWD_MAX_T, BF, None,
               lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, f32=False), _check_fwd(TOL_TC, "tc")),
    "tc.out_f32": (lambda T, c: T <= TC_FWD_MAX_T, BF, None,
                   lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, out=False), _check_fwd(TOL_TC, "tc")),
    "tc.both": (lambda T, c: T <= TC_FWD_MAX_T, BF, None,
                lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a), _check_fwd(TOL_TC, "tc")),
    "fwd_lse": (lambda T, c: TC_BWD_MAX_T < T <= TC_FWD_MAX_T, BF, None,   # (below: with the backward)
                lambda o, x, do, B, T, H, c, a: _run_lse(o, x, do, B, T, H, c, a, False), _check_lse(False)),
    "fwd_lse+bwd_lse": (lambda T, c: T <= TC_BWD_MAX_T, BF, BF,
                        lambda o, x, do, B, T, H, c, a: _run_lse(o, x, do, B, T, H, c, a, True), _check_lse(True)),
    "simt.f32": (lambda T, c: T <= SIMT_MAX_T, F32, None,
                 lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, split=True),
                 _check_fwd(TOL_F32, "simt_f32", split=True)),
    "simt.bf16": (lambda T, c: T <= SIMT_MAX_T, BF, None,
                  lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, split=True, simt=True),
                  _check_fwd(TOL_F32, "simt_bf16", split=True)),
    "row0.f32": (lambda T, c: not c, F32, None,
                 lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, split=True, row0=True),
                 _check_fwd(TOL_F32, "row0_f32", split=True, row0=True)),
    "row0.bf16": (lambda T, c: not c, BF, None,
                  lambda o, x, do, B, T, H, c, a: _fwd(o, x, B, T, H, c, a, split=True, row0=True),
                  _check_fwd(TOL_F32, "row0_bf16", split=True, row0=True)),
    "row0_bwd.f32": (lambda T, c: not c, F32, "row0", _run_row0_bwd, _check_row0_bwd("row0_bwd_f32.dqkv")),
    "row0_bwd.bf16": (lambda T, c: not c, BF, "row0", _run_row0_bwd, _check_row0_bwd("row0_bwd_bf16.dqkv")),
    "bwd.bf16_bf16_bf16": (lambda T, c: True, BF, BF,
                           lambda o, x, do, B, T, H, c, a: _run_bwd(o, x, do, B, T, H, c, a, BF),
                           _check_bwd("bwd_bf16.dqkv", TOL_BF16_BWD)),
    "bwd.bf16_f32_bf16": (lambda T, c: True, BF, F32,
                          lambda o, x, do, B, T, H, c, a: _run_bwd(o, x, do, B, T, H, c, a, BF),
                          _check_bwd("bwd_bf16_do_f32.dqkv", TOL_BF16_BWD, round_do=True)),
    "bwd.f32": (lambda T, c: simt_bwd_fits(T, F32), F32, F32,
                lambda o, x, do, B, T, H, c, a: _run_bwd(o, x, do, B, T, H, c, a, F32),
                _check_bwd("bwd_f32.dqkv", TOL_F32_BWD)),
}


def _inputs(kind, B, T, H, causal, seed, pad=0):
    """(qkv fp32, dO fp32) on the device; bf16 kernels get them rounded.  With `pad`, both are views of
    buffers with `pad` NaN columns and one NaN row after the last sequence."""
    d = H * 64
    g = torch.Generator().manual_seed(seed)
    if kind == "spiked":
        qkv = spiked_qkv(B, T, H, spike_pairs(T, causal), seed=seed, dtype=torch.float32)
    else:
        qkv = torch.randn(B * T, 3 * d, generator=g) * 0.7
    do = torch.randn(B * T, d, generator=g)
    if pad:
        qb = torch.full((B * T + 1, 3 * d + pad), float("nan"))
        qb[:B * T, :3 * d] = qkv
        db = torch.full((B * T + 1, d + pad), float("nan"))
        db[:B * T, :d] = do
        return qb.to(DEV)[:B * T, :3 * d], db.to(DEV)[:B * T, :d]
    return qkv.to(DEV), do.to(DEV)


def _cast(x, dtype, pad):
    """x in `dtype`, keeping a padded row stride (with its NaN padding) when `pad` is set."""
    if x.dtype == dtype:
        return x
    if not pad:
        return x.to(dtype)
    base = torch.full((x.shape[0] + 1, x.stride(0)), float("nan"), dtype=dtype, device=DEV)
    base[:x.shape[0], :x.shape[1]] = x.to(dtype)
    return base[:x.shape[0], :x.shape[1]]


def _run(ops, name, qkv32, do32, B, T, H, causal, alloc):
    accepts, qdt, ddt, run, check = KERNELS[name]
    pad = alloc.pad
    x = _cast(qkv32, qdt, pad)
    if ddt == "row0":
        do = do32.view(B, T, -1)[:, 0] if not pad else do32[::T]
    elif ddt is not None:
        do = _cast(do32, ddt, pad)
    else:
        do = None
    outs = run(ops, x, do, B, T, H, causal, alloc)
    torch.cuda.synchronize()
    return outs, (lambda: check(outs, x, do, B, T, H, causal))


# ---------------------------------------------------------------------------------------- T sweep
@pytest.mark.parametrize("kind", ["random", "spiked"])
@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("T", SWEEP_T)
def test_sweep(T, causal, kind):
    ops = _ops()
    B, H = 3, 2
    qkv, do = _inputs(kind, B, T, H, causal, seed=T * 2 + causal)
    for name, (accepts, *_rest) in KERNELS.items():
        if accepts(T, causal):
            _outs, check = _run(ops, name, qkv, do, B, T, H, causal, Alloc())
            check()


# ---------------------------------------------------------------------------------------- production shapes
@pytest.mark.parametrize("B,T,H,causal,names", [
    (32, 257, 16, False, ["tc.both"]),                              # CLIP ViT-L/14 vision
    (66, 77, 12, True, ["tc.both"]),                                # CLIP text
    (256, 197, 12, False, ["fwd_lse+bwd_lse"]),                     # ViT-B/16 training step
    (32, 65, 16, False, ["tc.both", "bwd.bf16_bf16_bf16"]),         # 112 px, general placement
    (32, 257, 16, False, ["row0_bwd.bf16"]),                        # bf16 CLIP step, last vision block
])
def test_production_shapes(B, T, H, causal, names):
    ops = _ops()
    qkv, do = _inputs("random", B, T, H, causal, seed=B + T)
    for name in names:
        outs, check = _run(ops, name, qkv, do, B, T, H, causal, Alloc())
        check()
        again, _ = _run(ops, name, qkv, do, B, T, H, causal, Alloc())
        for k in outs:
            assert torch.equal(outs[k], again[k]), (name, k, "repeated launch differs")


# ---------------------------------------------------------------------------------------- sequences
def _per_seq(t, B):
    return t.reshape(B, -1)


ISO_T = [77, 128, 197, 257]


@pytest.mark.parametrize("T", ISO_T)
def test_slicing_and_permutation_are_bit_exact(T):
    """Sequence b of a B-sequence launch equals a launch of that sequence alone, and permuting the
    sequences permutes the outputs, bit for bit (B * H = 192 units: CTAs own more than one)."""
    ops = _ops()
    B, H = 16, 12
    qkv, do = _inputs("random", B, T, H, False, seed=T)
    perm = torch.randperm(B, generator=torch.Generator().manual_seed(T)).tolist()
    rows = lambda x, idx: x.view(B, T, -1)[idx].reshape(len(idx) * T, -1)  # noqa: E731
    for name, (accepts, *_rest) in KERNELS.items():
        if not accepts(T, False):
            continue
        full, _ = _run(ops, name, qkv, do, B, T, H, False, Alloc())
        for b in (0, 7, B - 1):
            one, _ = _run(ops, name, rows(qkv, [b]), rows(do, [b]), 1, T, H, False, Alloc())
            for k in full:
                assert torch.equal(_per_seq(full[k], B)[b], _per_seq(one[k], 1)[0]), (name, k, b)
        pm, _ = _run(ops, name, rows(qkv, perm), rows(do, perm), B, T, H, False, Alloc())
        for k in full:
            assert torch.equal(_per_seq(pm[k], B), _per_seq(full[k], B)[perm]), (name, k, "permutation")


@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("T", ISO_T)
def test_sequence_isolation(T, causal):
    """NaN / +-Inf in rows 0..15 of sequence b+1 (Q, K, V and dO) leave every output of sequence b
    finite and bit-identical."""
    ops = _ops()
    B, H = 4, 2
    qkv, do = _inputs("random", B, T, H, causal, seed=T + 1)
    bad = torch.tensor([float("nan"), float("inf"), float("-inf")], device=DEV)
    qkv_p, do_p = qkv.clone(), do.clone()
    for b in (1, 3):
        for x in (qkv_p, do_p):
            blk = x[b * T:b * T + 16]
            idx = torch.arange(blk.numel(), device=DEV).view_as(blk) % 3
            blk.copy_(bad[idx])
    for name, (accepts, *_rest) in KERNELS.items():
        if not accepts(T, causal):
            continue
        clean, _ = _run(ops, name, qkv, do, B, T, H, causal, Alloc())
        dirty, _ = _run(ops, name, qkv_p, do_p, B, T, H, causal, Alloc())
        for k in clean:
            c, p = _per_seq(clean[k], B), _per_seq(dirty[k], B)
            for b in (0, 2):
                assert bool(torch.isfinite(p[b].float()).all()), (name, k, b, "non-finite leaked in")
                assert torch.equal(c[b], p[b]), (name, k, b)


# ---------------------------------------------------------------------------------------- layouts
@pytest.mark.parametrize("causal", [False, True])
@pytest.mark.parametrize("T", [77, 257])
def test_layout_canaries(T, causal):
    """ld_qkv = 3d + 8, ld_out = d + 8, ld_of = d + 4 (dO and bf16 dQKV likewise padded by 8, fp32
    dQKV by 4), NaN in the input padding and a trailing NaN row: every in-range element is written
    correctly and nothing outside the logical outputs is."""
    ops = _ops()
    B, H = 3, 2
    qkv, do = _inputs("random", B, T, H, causal, seed=T + 5, pad=8)
    for name, (accepts, *_rest) in KERNELS.items():
        if not accepts(T, causal):
            continue
        alloc = Alloc(pad=8)
        _outs, check = _run(ops, name, qkv, do, B, T, H, causal, alloc)
        check()
        alloc.assert_outside_untouched()


# ---------------------------------------------------------------------------------------- rejection
def _expect_arg_error(fn, *untouched):
    before = [t.clone() for t in untouched]
    with pytest.raises(RuntimeError, match=rf"code {HBA_ERR_ARG}\)"):
        fn()
    torch.cuda.synchronize()
    for t, b in zip(untouched, before):
        assert torch.equal(t, b), "a rejected call wrote its output"


def test_rejections_leave_the_library_usable():
    ops = _ops()
    H, d = 1, 64
    for T in (289, 258, 257, 204):
        qkv, do = _inputs("random", 1, T, H, False, seed=T)
        qb, db = qkv.to(BF), do.to(BF)
        out = torch.full((T, d), SENTINEL, device=DEV, dtype=BF)
        of = torch.full((T, d), SENTINEL, device=DEV)
        lse = torch.full((H * T,), SENTINEL, device=DEV)
        dqb = torch.full((T, 3 * d), SENTINEL, device=DEV, dtype=BF)
        dqf = torch.full((T, 3 * d), SENTINEL, device=DEV)
        if T == 289:
            for x in (qkv, qb):
                _expect_arg_error(lambda: ops.attention_fwd(x, 1, T, H, out=ops.Operand(out, T, d, 0), out_f32=of),
                                  out, of)
                _expect_arg_error(lambda: ops.attention_fwd(x, 1, T, H, first_row_only=True, out_f32=of), of)
                _expect_arg_error(lambda: ops.attention_bwd_row0(x, 1, T, H, do[:1], dqf), dqf)
            _expect_arg_error(lambda: ops.attention_bwd(qb, 1, T, H, db, dqb), dqb)
            _expect_arg_error(lambda: ops.attention_bwd(qkv, 1, T, H, do, dqf), dqf)
        if T in (289, 258):
            _expect_arg_error(lambda: ops.attention_fwd_lse(qb, 1, T, H, out, lse), out, lse)
        if T in (289, 258, 257):
            _expect_arg_error(lambda: ops.attention_bwd_lse(qb, 1, T, H, out, db, lse, dqb), dqb)
        if T == 204:   # fp32 tiles of 204 rows exceed 227 KB of shared memory
            _expect_arg_error(lambda: ops.attention_bwd(qkv, 1, T, H, do, dqf), dqf)
    T = 77
    qkv, do = _inputs("random", 2, T, H, False, seed=3)
    of = torch.full((2, d), SENTINEL, device=DEV)
    _expect_arg_error(lambda: ops.attention_fwd(qkv.to(BF), 2, T, H, causal=True, first_row_only=True, out_f32=of),
                      of)
    # the library still works after the rejections
    for name in ("tc.both", "fwd_lse+bwd_lse", "bwd.f32"):
        _outs, check = _run(ops, name, qkv, do, 2, T, H, True, Alloc())
        check()
