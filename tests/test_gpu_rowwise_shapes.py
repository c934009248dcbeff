"""The row-wise kernels (LayerNorm forward in both forms, backward, fused backward, parameter gradients, column sums,
token assembly, operand staging, row helpers) at every launch branch, against the fp64 references of
tests/rowwise_ref.py, element by element.

Every output element is checked as |out - ref| <= bound, with the bound of tests/rowwise_ref.py (derivation in its
docstring): an fp32 error analysis of the kernels' own arithmetic - the lane-partial-then-shuffle sums of the mean,
the centred sum of squares and s1 / s2, 2 ulp of rsqrtf, the chunked column sums, one rounding of the stored type -
absolute per row through the mean's error, so that a constant row or a row with |mean| / sigma = 2^10 is held to
what the kernel can actually reach, and a wrong mean, variance or dropped row moves elements far past it.  The worst
|out - ref| / bound by path is printed at the end of the module.

Also: NaN canvases around every output (padded leading dimensions, the gap between hi and lo columns, rows past
`rows`, rows skipped by a row step), NaN in the input padding, bit-exact properties (bf16 outputs = split of the f32
output; streaming = per-row LayerNorm forward; row slices and permutations; accumulate = fp32(plain + prev);
repeated launches), the production shapes of both trainers and argument rejection."""
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from rowwise_ref import (EPS_CLIP, EPS_TIMM, FUSED_COLS, assemble_x, bwd_dy,  # noqa: E402
                         colsum_bound, fused_depth, ln_bwd_bound, ln_bwd_ref, ln_fwd_bound, ln_fwd_branches,
                         ln_fwd_ref, ln_params, ln_rows, param_grad_bound, param_grad_ref, strided, wrap_rows)

pytestmark = pytest.mark.gpu

DEV = "cuda"
HBA_ERR_ARG = -22
NAN = float("nan")
WORST = {}   # path -> worst |out - ref| / bound over the module


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst |out - ref| / bound by path (tolerance 1):")
        for k in sorted(WORST):
            print(f"  {k:40s} {WORST[k]:.3e}")


def _ops():
    import hba  # noqa: F401
    from hba import ops
    return ops


def _sync():
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------- buffers
def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32)


class Canvas:
    """Output buffers filled with NaN (bf16: 0x7fc0); `mask` marks the logical output.  `untouched()` asserts that
    nothing outside it changed."""

    def __init__(self):
        self.bufs = []

    def __call__(self, nrows, ld, dtype, regions, rows=None, init=None):
        buf = torch.full((nrows + 2, ld), NAN, dtype=dtype, device=DEV)
        mask = torch.zeros(buf.shape, dtype=torch.bool, device=DEV)
        sel = slice(0, nrows) if rows is None else rows
        for c0, w in regions:
            mask[sel, c0:c0 + w] = True
        if init is not None:
            buf[sel, :init.shape[1]] = init.to(DEV, dtype)
        self.bufs.append((buf, mask, buf.clone()))
        return buf

    def untouched(self, what=""):
        for buf, mask, init in self.bufs:
            assert torch.equal(_bits(buf)[~mask], _bits(init)[~mask]), f"{what}: write outside the logical output"


def _padded(x, ld_extra=4, row_step=1):
    """x [rows, cols] as rows r * row_step of a NaN-filled [rows * row_step + 1, cols + ld_extra] buffer (the view
    ends at the last logical row)."""
    rows, cols = x.shape
    buf = torch.full((rows * row_step + 1, cols + ld_extra), NAN, dtype=x.dtype, device=DEV)
    buf[:rows * row_step:row_step, :cols] = x.to(DEV)
    return buf[:(rows - 1) * row_step + 1, :cols]


def _vec(v, extra=4):
    buf = torch.full((v.numel() + extra,), NAN, dtype=v.dtype, device=DEV)
    buf[:v.numel()] = v.to(DEV)
    return buf[:v.numel()]


def _split(y):
    hi = y.to(torch.bfloat16)
    return hi, (y - hi.float()).to(torch.bfloat16)


def _record(path, got, ref, bnd, what):
    d = (got.double() - ref).abs()
    ratio = torch.where(bnd > 0, d / bnd.clamp_min(1e-300), torch.where(d == 0, 0.0, float("inf")))
    ratio = torch.where(torch.isnan(d), float("inf"), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    WORST[path] = max(WORST.get(path, 0.0), worst)
    if not worst <= 1.0:
        idx = int(ratio.flatten().argmax())
        cols = ratio.shape[-1] if ratio.dim() > 1 else ratio.numel()
        raise AssertionError(f"{what} {path}: |out - ref| / bound = {worst:.3g} at [{idx // cols}, {idx % cols}]: got "
                             f"{float(got.flatten()[idx])!r}, ref {float(ref.flatten()[idx])!r}, "
                             f"bound {float(bnd.flatten()[idx]):.3g}")


OUTS = (("f32",), ("bf16",), ("hilo",), ("f32", "hilo"), ("f32", "bf16"))


def _outputs(cv, ops, rows, cols, outs):
    """NaN-canvas outputs of one LayerNorm-like call: f32 [rows, cols + 4]; bf16 hi at [0, cols), lo (hilo) at
    [cols + 8, 2 cols + 8) with a gap between them."""
    o = {}
    if "f32" in outs:
        o["f32"] = cv(rows, cols + 4, torch.float32, [(0, cols)])
    bf = "hilo" if "hilo" in outs else ("bf16" if "bf16" in outs else None)
    if bf:
        lo = cols + 8 if bf == "hilo" else 0
        buf = cv(rows, 2 * cols + 12, torch.bfloat16, [(0, cols)] + ([(lo, cols)] if lo else []))
        o["op"] = ops.Operand(buf, rows, cols, lo)
    return o, bf


def _check_outputs(path, o, bf, rows, cols, ref, bound_fn, what):
    """Per-element check of every output form, and the bf16 parts = split of the f32 output of the same call."""
    got = {}
    if "f32" in o:
        got["f32"] = o["f32"][:rows, :cols]
        _record(f"{path}.f32", got["f32"], ref, bound_fn("f32"), what)
    if bf:
        op = o["op"]
        hi = op.buf[:rows, :cols]
        got["hi"] = hi
        val = hi.float() + (op.buf[:rows, op.lo_off:op.lo_off + cols].float() if op.lo_off else 0)
        _record(f"{path}.{bf}", val, ref, bound_fn(bf), what)
        if op.lo_off:
            got["lo"] = op.buf[:rows, op.lo_off:op.lo_off + cols]
        if "f32" in got:
            h, lo = _split(got["f32"])
            assert torch.equal(_bits(hi), _bits(h)), f"{what}: bf16 hi != split(y_f32)"
            if op.lo_off:
                assert torch.equal(_bits(got["lo"]), _bits(lo)), f"{what}: bf16 lo != split(y_f32)"
    return got


# ---------------------------------------------------------------------------------------- one checked call each
def ln_fwd_case(ops, rows, cols, *, row_step=1, outs=("f32",), eps=EPS_CLIP, seed=0, x=None, params=None, check=True):
    x = ln_rows(rows, cols, seed, eps) if x is None else x
    gamma, beta = ln_params(cols, seed) if params is None else params
    xs = _padded(x, row_step=row_step)
    g, b = _vec(gamma), _vec(beta)
    cv = Canvas()
    o, bf = _outputs(cv, ops, rows, cols, outs)
    ops.layernorm_fwd(xs, rows, cols, g, b, eps, row_step=row_step, y_f32=o["f32"][:rows, :cols] if "f32" in o else None,
                      y=o.get("op"))
    _sync()
    what = f"ln_fwd rows={rows} cols={cols} row_step={row_step} outs={outs} eps={eps}"
    cv.untouched(what)
    if not check:
        return {"f32": o["f32"][:rows, :cols]} if "f32" in o else {"op": o["op"].buf[:rows]}
    st = ln_fwd_ref(x.to(DEV), gamma.to(DEV), beta.to(DEV), eps)
    form = ln_fwd_branches(rows, cols)["form"]
    return _check_outputs(f"ln_fwd.{form}", o, bf, rows, cols, st["y"], lambda out: ln_fwd_bound(st, out), what)


def ln_bwd_case(ops, rows, cols, *, row_step=1, accumulate=False, eps=EPS_CLIP, seed=0, check=True):
    x = ln_rows(rows, cols, seed, eps)
    gamma, _ = ln_params(cols, seed, zeros=False)
    dy = bwd_dy(x, gamma, eps, seed)
    prev = torch.randn(rows, cols, generator=torch.Generator().manual_seed(seed + 3)) * 4 if accumulate else None
    xs, dys, g = _padded(x, row_step=row_step), _padded(dy), _vec(gamma)
    cv = Canvas()
    dx = cv(rows, cols + 4, torch.float32, [(0, cols)], init=prev)
    ops.layernorm_bwd(dys, xs, rows, cols, g, eps, dx[:rows, :cols], row_step=row_step, accumulate=accumulate)
    _sync()
    what = f"ln_bwd rows={rows} cols={cols} row_step={row_step} accumulate={accumulate} eps={eps}"
    cv.untouched(what)
    out = dx[:rows, :cols]
    if check:
        st = ln_bwd_ref(dy.to(DEV), x.to(DEV), gamma.to(DEV), eps, prev.to(DEV) if prev is not None else None)
        _record("ln_bwd" + (".acc" if accumulate else ""), out, st["dx"], ln_bwd_bound(st), what)
    return out, (x, dy, gamma, prev)


def bwd_fused_case(ops, rows, cols, *, accumulate=False, accumulate_params=False, bf=None, colsum=True, eps=EPS_TIMM,
                   seed=0, x=None, check=True):
    x = ln_rows(rows, cols, seed, eps) if x is None else x
    gamma, _ = ln_params(cols, seed, zeros=False)
    dy = bwd_dy(x, gamma, eps, seed)
    gen = torch.Generator().manual_seed(seed + 5)
    prev = torch.randn(rows, cols, generator=gen) * 4 if accumulate else None
    prev_p = torch.randn(2 * cols, generator=gen) * 50 if accumulate_params else None
    xs, dys, g = _padded(x), _padded(dy), _vec(gamma)
    cv = Canvas()
    dx = cv(rows, cols + 4, torch.float32, [(0, cols)], init=prev)
    o, bfk = _outputs(cv, ops, rows, cols, (bf,) if bf else ())
    dgb = cv(1, 2 * cols + 4, torch.float32, [(0, 2 * cols)], init=prev_p[None] if prev_p is not None else None)
    cs = cv(1, cols + 4, torch.float32, [(0, cols)]) if colsum else None
    ws = torch.full((2 * 148 * 3 * cols,), NAN, device=DEV)
    ops.layernorm_bwd_fused(dys, xs, rows, cols, g, eps, dx[:rows, :cols], dgb[0, :2 * cols], ws,
                            accumulate=accumulate, dx_op=o.get("op"), dx_colsum=cs[0, :cols] if colsum else None,
                            accumulate_params=accumulate_params)
    _sync()
    what = f"bwd_fused rows={rows} cols={cols} accumulate={accumulate}/{accumulate_params} bf={bf} colsum={colsum}"
    cv.untouched(what)
    got = {"dx": dx[:rows, :cols], "dgb": dgb[0, :2 * cols]}
    if colsum:
        got["cs"] = cs[0, :cols]
    if bfk:
        got["hi"] = o["op"].buf[:rows, :cols]
        h, lo = _split(got["dx"])
        assert torch.equal(_bits(got["hi"]), _bits(h)), f"{what}: bf16 hi != split(dx)"
        if o["op"].lo_off:
            got["lo"] = o["op"].buf[:rows, o["op"].lo_off:o["op"].lo_off + cols]
            assert torch.equal(_bits(got["lo"]), _bits(lo)), f"{what}: bf16 lo != split(dx)"
    if not check:
        return got
    dv, xv, gv = dy.to(DEV), x.to(DEV), gamma.to(DEV)
    st = ln_bwd_ref(dv, xv, gv, eps, prev.to(DEV) if prev is not None else None)
    _record("bwd_fused.dx" + (".acc" if accumulate else ""), got["dx"], st["dx"], ln_bwd_bound(st, fused=True), what)
    D = fused_depth(rows)
    if bfk:
        val = got["hi"].float() + (got["lo"].float() if "lo" in got else 0)
        _record(f"bwd_fused.{bfk}", val, st["dx"], ln_bwd_bound(st, fused=True, out=bfk), what)
    ref, bnd = param_grad_bound(param_grad_ref(dv, xv, eps), prev_p.to(DEV) if prev_p is not None else None, D=D,
                                fused=True)
    _record("bwd_fused.dgamma_dbeta" + (".acc" if accumulate_params else ""), got["dgb"], ref, bnd, what)
    if colsum:   # the column sums of the kernel's own dx (after accumulation)
        ref, bnd = colsum_bound(got["dx"], D=D)
        _record("bwd_fused.dx_colsum", got["cs"], ref, bnd, what)
    return got


def param_grad_case(ops, rows, cols, *, row_step=1, accumulate=False, ld_extra=4, eps=EPS_TIMM, seed=0, check=True):
    x = torch.randn(rows, cols, generator=torch.Generator().manual_seed(seed)) * 2 + 0.5
    if cols % 128 == 0:
        x = ln_rows(rows, cols, seed, eps)
    dy = torch.randn(rows, cols, generator=torch.Generator().manual_seed(seed + 1)) * 3
    prev = torch.randn(2 * cols, generator=torch.Generator().manual_seed(seed + 2)) * 50 if accumulate else None
    xs, dys = _padded(x, ld_extra=ld_extra, row_step=row_step), _padded(dy, ld_extra=ld_extra + 3)
    cv = Canvas()
    out = cv(1, 2 * cols + 4, torch.float32, [(0, 2 * cols)], init=prev[None] if prev is not None else None)
    ws = torch.full((2 * rows + 256 * cols + 64,), NAN, device=DEV)
    ops.layernorm_param_grad(dys, xs, rows, cols, eps, out[0, :2 * cols], ws, row_step=row_step, accumulate=accumulate)
    _sync()
    what = f"param_grad rows={rows} cols={cols} row_step={row_step} accumulate={accumulate} ldx={xs.stride(0)}"
    cv.untouched(what)
    got = out[0, :2 * cols]
    if check:
        ref, bnd = param_grad_bound(param_grad_ref(dy.to(DEV), x.to(DEV), eps), prev.to(DEV) if prev is not None else None)
        _record("param_grad" + (".acc" if accumulate else ""), got, ref, bnd, what)
    return got


def colsum_case(ops, rows, cols, dtype, *, accumulate=False, ld_extra=4, seed=0, check=True, x=None):
    if x is None:
        g = torch.Generator().manual_seed(seed)
        x = torch.randn(rows, cols, generator=g) * torch.exp2(torch.randint(-8, 9, (rows, 1), generator=g).float())
        x = x.to(dtype)
    prev = torch.randn(cols, generator=torch.Generator().manual_seed(seed + 9)) * 100 if accumulate else None
    xs = _padded(x, ld_extra=ld_extra)
    cv = Canvas()
    out = cv(1, cols + 4, torch.float32, [(0, cols)], init=prev[None] if prev is not None else None)
    ws = torch.full((128 * cols + 64,), NAN, device=DEV)
    ops.colsum(xs, out[0, :cols], ws, accumulate=accumulate)
    _sync()
    what = f"colsum rows={rows} cols={cols} {dtype} accumulate={accumulate} ld={xs.stride(0)}"
    cv.untouched(what)
    got = out[0, :cols]
    if check:
        ref, bnd = colsum_bound(x.to(DEV), prev.to(DEV) if prev is not None else None)
        _record(f"colsum.{'bf16' if dtype == torch.bfloat16 else 'f32'}", got, ref, bnd, what)
    return got


# ---------------------------------------------------------------------------------------- LayerNorm forward sweep
SWEEP_COLS = [128, 256, 384, 512, 640, 768, 896, 1024]
EDGE_ROWS = [1, 7, 8, 9, 1023, 1024, 1025, 3551, 3552, 3553]


def fwd_rows(cols):
    return EDGE_ROWS + [wrap_rows(cols, 1), wrap_rows(cols, 2)]


@pytest.mark.parametrize("cols", SWEEP_COLS)
def test_ln_fwd_sweep(cols):
    """Every row count of fwd_rows(cols) (per-row kernel, streaming grid below / at 148, one or several iterations,
    ring wraps, partial last stages), every output form in turn, both eps values."""
    ops = _ops()
    for i, rows in enumerate(fwd_rows(cols)):
        ln_fwd_case(ops, rows, cols, outs=OUTS[i % len(OUTS)], eps=(EPS_CLIP, EPS_TIMM)[i % 2], seed=rows + cols)


@pytest.mark.parametrize("row_step", [1, 3])
@pytest.mark.parametrize("cols", SWEEP_COLS)
def test_ln_fwd_streaming_equals_per_row(cols, row_step):
    """The streaming form (>= 1024 rows) gives the bits of the per-row kernel run on the same rows in chunks of < 1024
    rows, at every cols and row step; includes the shapes of the CLIP-HBA step (8224 x 1024, 5082 x 768)."""
    ops = _ops()
    shapes = {1024: [8224, 3000, 1025], 768: [5082, 1024], 128: [1024, 3553], 256: [1031, 3552]}.get(cols, [1025, 3553])
    for rows in shapes:
        x = ln_rows(rows, cols, seed=rows)
        params = ln_params(cols, rows)
        full = ln_fwd_case(ops, rows, cols, row_step=row_step, outs=("f32", "hilo"), x=x, seed=rows, params=params)
        xs = _padded(strided(x, row_step, rows))
        g, b = _vec(params[0]), _vec(params[1])
        yc = torch.full((rows, cols), NAN, device=DEV)
        for r0 in range(0, rows, 1000):
            n = min(1000, rows - r0)
            ops.layernorm_fwd(xs[r0 * row_step:], n, cols, g, b, EPS_CLIP, row_step=row_step, y_f32=yc[r0:])
        _sync()
        assert torch.equal(_bits(yc), _bits(full["f32"])), (rows, cols, row_step)


@pytest.mark.parametrize("cols", SWEEP_COLS)
def test_ln_fwd_row_step(cols):
    """row_step > 1 in both forms (the CLS rows of every image): rows skipped by the step are never read (NaN there)."""
    ops = _ops()
    for rows, step, outs in ((9, 3, ("f32", "bf16")), (1025, 3, ("hilo",)), (3553, 2, ("f32", "hilo"))):
        x = ln_rows(rows, cols, seed=step)
        ln_fwd_case(ops, rows, cols, row_step=step, outs=outs, x=x, seed=step)


# ---------------------------------------------------------------------------------------- backward
BWD_ROWS = [1, 7, 8, 9, 1023, 1025, 3553]


@pytest.mark.parametrize("cols", SWEEP_COLS)
def test_ln_bwd_sweep(cols):
    """LN backward at every cols, row step 1 and 3, accumulate on and off; accumulate = fp32(plain + prev) exactly."""
    ops = _ops()
    for i, rows in enumerate(BWD_ROWS):
        step = 3 if i % 2 else 1
        eps = (EPS_CLIP, EPS_TIMM)[i % 2]
        plain, _ = ln_bwd_case(ops, rows, cols, row_step=step, eps=eps, seed=rows)
        acc, (_, _, _, prev) = ln_bwd_case(ops, rows, cols, row_step=step, accumulate=True, eps=eps, seed=rows)
        assert torch.equal(_bits(acc), _bits(plain + prev.to(DEV))), (rows, cols, step)


FUSED_ROWS = [1, 7, 9, 1023, 2368, 2369, 8000]       # one row per warp up to 8 x 296 = 2368 rows, several above


@pytest.mark.parametrize("cols", FUSED_COLS)
def test_bwd_fused_sweep(cols):
    """Every NVEC, one and several rows per warp, with and without accumulate / accumulate_params / dx_colsum / the
    bf16 copy (hi only, hi + lo); accumulate and accumulate_params give fp32(plain + prev) exactly."""
    ops = _ops()
    for i, rows in enumerate(FUSED_ROWS):
        bf = (None, "bf16", "hilo")[i % 3]
        cs = i % 2 == 0
        plain = bwd_fused_case(ops, rows, cols, bf=bf, colsum=cs, seed=rows)
        acc = bwd_fused_case(ops, rows, cols, accumulate=True, accumulate_params=True, bf=bf, colsum=not cs, seed=rows)
        gen = torch.Generator().manual_seed(rows + 5)
        prev = torch.randn(rows, cols, generator=gen) * 4
        prev_p = torch.randn(2 * cols, generator=gen) * 50
        assert torch.equal(_bits(acc["dx"]), _bits(plain["dx"] + prev.to(DEV))), (rows, cols)
        assert torch.equal(_bits(acc["dgb"]), _bits(plain["dgb"] + prev_p.to(DEV))), (rows, cols)


# ---------------------------------------------------------------------------------------- column sums
PG_SHAPES = [(1, 128), (7, 100), (127, 768), (129, 36), (300, 768), (1000, 1000), (5000, 1024)]


@pytest.mark.parametrize("rows,cols", PG_SHAPES)
def test_param_grad(rows, cols):
    """Empty chunks (rows < 128 and 129), a partial column block (cols % 32 != 0), row_step 1 / 197, ldx > cols,
    accumulate on and off (accumulate = fp32(plain + prev) exactly); repeated launches give the same bits."""
    ops = _ops()
    for step in (1, 197 if rows <= 300 else 2):
        plain = param_grad_case(ops, rows, cols, row_step=step, seed=rows + step)
        acc = param_grad_case(ops, rows, cols, row_step=step, accumulate=True, ld_extra=8, seed=rows + step)
        prev = torch.randn(2 * cols, generator=torch.Generator().manual_seed(rows + step + 2)) * 50
        assert torch.equal(_bits(acc), _bits(plain + prev.to(DEV)))
        again = param_grad_case(ops, rows, cols, row_step=step, seed=rows + step, check=False)
        assert torch.equal(_bits(again), _bits(plain))


CS_SHAPES = [(1, 128), (9, 33), (127, 100), (129, 768), (777, 1000), (5120, 36), (50432, 768)]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("rows,cols", CS_SHAPES)
def test_colsum(rows, cols, dtype):
    ops = _ops()
    plain = colsum_case(ops, rows, cols, dtype, seed=rows)
    acc = colsum_case(ops, rows, cols, dtype, accumulate=True, ld_extra=12, seed=rows)
    prev = torch.randn(cols, generator=torch.Generator().manual_seed(rows + 9)) * 100
    assert torch.equal(_bits(acc), _bits(plain + prev.to(DEV)))
    assert torch.equal(_bits(colsum_case(ops, rows, cols, dtype, seed=rows, check=False)), _bits(plain))


# ---------------------------------------------------------------------------------------- row-local bit properties
def _bwd_dx(ops, fused, dy, x, gamma):
    rows, cols = x.shape
    dx = torch.full((rows, cols), NAN, device=DEV)
    if fused:
        ops.layernorm_bwd_fused(dy.to(DEV), x.to(DEV), rows, cols, gamma.to(DEV), EPS_TIMM, dx,
                                torch.empty(2 * cols, device=DEV), torch.empty(2 * 148 * 3 * cols, device=DEV))
    else:
        ops.layernorm_bwd(dy.to(DEV), x.to(DEV), rows, cols, gamma.to(DEV), EPS_TIMM, dx)
    _sync()
    return dx


def test_row_slices_and_permutations_are_bit_exact():
    """LN forward (both forms), LN backward and bwd_fused's dx on a row slice or a row permutation give the bits of
    the full call's rows: a row's result does not depend on its place in the grid."""
    ops = _ops()
    cols = 768
    for rows in (300, 3553):
        x = ln_rows(rows, cols, seed=1)
        perm = torch.randperm(rows, generator=torch.Generator().manual_seed(2))
        full = ln_fwd_case(ops, rows, cols, outs=("f32",), x=x, seed=1)["f32"]
        pf = ln_fwd_case(ops, rows, cols, outs=("f32",), x=x[perm], seed=1, check=False)["f32"]
        assert torch.equal(_bits(pf), _bits(full[perm.to(DEV)]))
        for r0, n in ((0, 1), (37, 200), (rows - 9, 9)):
            part = ln_fwd_case(ops, n, cols, outs=("f32",), x=x[r0:r0 + n], seed=1, check=False)["f32"]
            assert torch.equal(_bits(part), _bits(full[r0:r0 + n])), (rows, r0, n)
    rows = 2500                                      # bwd_fused: 296 blocks, several rows per warp
    x = ln_rows(rows, cols, seed=3)
    gamma, _ = ln_params(cols, 3, zeros=False)
    dy = bwd_dy(x, gamma, EPS_TIMM, 3)
    perm = torch.randperm(rows, generator=torch.Generator().manual_seed(4))
    for fused in (False, True):
        full = _bwd_dx(ops, fused, dy, x, gamma)
        assert torch.equal(_bits(_bwd_dx(ops, fused, dy[perm], x[perm], gamma)), _bits(full[perm.to(DEV)])), fused
        assert torch.equal(_bits(_bwd_dx(ops, fused, dy[100:200], x[100:200], gamma)), _bits(full[100:200])), fused


# ---------------------------------------------------------------------------------------- staging and helpers
def test_add_rows_and_gather_rows_match_torch():
    ops = _ops()
    g = torch.Generator().manual_seed(11)
    for rows, cols, step in ((1, 1, 1), (37, 45, 3), (300, 768, 197), (9, 1000, 1)):
        src = _padded(torch.randn(rows, cols, generator=g), ld_extra=5)
        cv = Canvas()
        sel = torch.zeros(rows * step + 2, dtype=torch.bool, device=DEV)
        sel[:rows * step:step] = True            # the rows between are skipped and must stay NaN
        dst = cv(rows * step, cols + 7, torch.float32, [(0, cols)], rows=sel, init=torch.randn(rows, cols, generator=g))
        want = dst.clone()
        want[sel, :cols] += src
        ops.add_rows(dst[:, :cols], src, rows, cols, dst_row_step=step)
        _sync()
        cv.untouched(f"add_rows {rows} {cols} {step}")
        assert torch.equal(_bits(dst), _bits(want)), (rows, cols, step)
        idx = torch.randint(0, rows, (2 * rows + 3,), generator=g).to(DEV)
        cv = Canvas()
        out = cv(idx.numel(), cols + 3, torch.float32, [(0, cols)])
        ops.gather_rows(src, idx, cols, out)
        _sync()
        cv.untouched("gather_rows")
        assert torch.equal(_bits(out[:idx.numel(), :cols]), _bits(src[idx]))


@pytest.mark.parametrize("transpose", [False, True])
def test_split_bf16_matches_round_to_nearest(transpose):
    ops = _ops()
    g = torch.Generator().manual_seed(12)
    for rows, cols in ((45, 76), (1, 4), (33, 36), (100, 300)):
        x = torch.randn(rows, cols, generator=g) * torch.exp2(torch.randint(-20, 21, (rows, cols), generator=g).float())
        xs = _padded(x, ld_extra=8)
        orows, ocols = (cols, rows) if transpose else (rows, cols)
        for lo in (0, ocols + 6):
            cv = Canvas()
            ld = (lo if lo else ocols) + ocols + 10
            buf = cv(orows, ld, torch.bfloat16, [(0, ocols)] + ([(lo, ocols)] if lo else []))
            ops.split_bf16(xs, ops.Operand(buf, orows, ocols, lo), transpose=transpose)
            _sync()
            cv.untouched(f"split_bf16 {rows}x{cols} lo={lo} T={transpose}")
            h, l = _split(x.t().contiguous() if transpose else x)
            assert torch.equal(_bits(buf[:orows, :ocols]), _bits(h.to(DEV)))
            if lo:
                assert torch.equal(_bits(buf[:orows, lo:lo + ocols]), _bits(l.to(DEV)))


@pytest.mark.parametrize("layout", ["hi_only", "operand", "tight_lo"])
def test_im2col_is_exact_and_zero_fills_the_padding(layout):
    """im2col = the conv's patch matrix (column c P^2 + py P + px), bit for bit, zeros in the pad columns of both
    parts, nothing past ld_out (tight_lo: the lo part ends before 2 lo_off)."""
    ops = _ops()
    B, H, W, P = 2, 48, 32, 16
    kk = 3 * P * P
    img = torch.randn(B, 3, H, W, generator=torch.Generator().manual_seed(13))
    cols = img.view(B, 3, H // P, P, W // P, P).permute(0, 2, 4, 1, 3, 5).reshape(-1, kk)
    n = cols.shape[0]
    lo, ld = {"hi_only": (0, kk + 40), "operand": (kk + 16, 2 * kk + 32), "tight_lo": (kk + 24, 2 * kk + 32)}[layout]
    cv = Canvas()
    buf = cv(n, ld, torch.bfloat16, [(0, ld)])
    ops.im2col_patches(img.to(DEV), P, ops.Operand(buf[:n], n, kk, lo))
    _sync()
    cv.untouched(f"im2col {layout}")
    h, l = _split(cols)
    want = torch.zeros(n, ld, dtype=torch.bfloat16)
    want[:, :kk] = h
    if lo:
        want[:, lo:lo + kk] = l
    assert torch.equal(_bits(buf[:n]), _bits(want.to(DEV)))


def test_assemble_tokens_with_and_without_ln_pre():
    ops = _ops()
    g = torch.Generator().manual_seed(14)
    for B, npatch, width, eps in ((3, 49, 768, EPS_TIMM), (2, 256, 1024, EPS_CLIP), (1, 4, 128, EPS_CLIP)):
        conv = torch.randn(B * npatch, width, generator=g) * 3
        conv[::5] += 200.0                                   # rows with a large offset
        cls = torch.randn(width, generator=g)
        pos = torch.randn(npatch + 1, width, generator=g)
        gamma, beta = ln_params(width, B)
        xa = assemble_x(conv, cls, pos, B, npatch)
        for ln in (False, True):
            cv = Canvas()
            out = cv(B * (npatch + 1), width, torch.float32, [(0, width)])
            ops.assemble_tokens_ln(conv.to(DEV), B, npatch, width, cls.to(DEV), pos.to(DEV),
                                   gamma.to(DEV) if ln else None, beta.to(DEV) if ln else None, eps, out)
            _sync()
            cv.untouched("assemble")
            got = out[:B * (npatch + 1)]
            if ln:
                st = ln_fwd_ref(xa.to(DEV), gamma.to(DEV), beta.to(DEV), eps)
                _record("assemble.ln_pre", got, st["y"], ln_fwd_bound(st), f"assemble B={B} width={width}")
            else:
                assert torch.equal(_bits(got), _bits(xa.to(DEV)))


def test_nonfinite_flag():
    """Set by a NaN, +Inf or -Inf at the first or last element or past one grid-stride pass (592 x 256 elements);
    0 when every element is finite (a NaN just past n is not read)."""
    ops = _ops()
    n = 592 * 256 * 2 + 37
    base = torch.randn(n + 1, generator=torch.Generator().manual_seed(15)).to(DEV)
    base[n] = NAN
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.nonfinite_flag(base[:n], flag)
    _sync()
    assert int(flag) == 0
    for pos in (0, n - 1, 592 * 256 + 5):
        for bad in (NAN, float("inf"), float("-inf")):
            x = base.clone()
            x[pos] = bad
            flag.zero_()
            ops.nonfinite_flag(x[:n], flag)
            _sync()
            assert int(flag) == 1, (pos, bad)


# ---------------------------------------------------------------------------------------- production shapes
def test_production_shapes():
    """The row-wise calls of one training step of each trainer, with per-element bounds: CLIP-HBA ln_1 / ln_2 on
    8224 x 1024 and 5082 x 768 (hi + lo in fp32 mode, hi only in bf16 mode) and their backward (accumulating), the CLS
    rows of 32 images at row step 257; ViT-B/16 at batch 256: LN forward and bwd_fused on 50432 x 768, the CLS rows at
    row step 197 (forward, backward, parameter gradients) and the positional-embedding gradient, colsum of
    256 x 151296."""
    ops = _ops()
    for rows, cols in ((8224, 1024), (5082, 768)):
        ln_fwd_case(ops, rows, cols, outs=("hilo",), seed=1)
        ln_fwd_case(ops, rows, cols, outs=("bf16",), seed=2)
        ln_bwd_case(ops, rows, cols, accumulate=True, seed=3)
    ln_fwd_case(ops, 32, 1024, row_step=257, outs=("f32",), x=ln_rows(32, 1024, 4), seed=4)
    ln_bwd_case(ops, 32, 1024, row_step=257, seed=5)
    ln_fwd_case(ops, 50432, 768, outs=("bf16",), eps=EPS_TIMM, seed=6)
    ln_fwd_case(ops, 256, 768, row_step=197, outs=("hilo",), eps=EPS_TIMM, x=ln_rows(256, 768, 7), seed=7)
    ln_bwd_case(ops, 256, 768, row_step=197, eps=EPS_TIMM, seed=8)
    param_grad_case(ops, 256, 768, row_step=197, seed=9)
    bwd_fused_case(ops, 50432, 768, accumulate=True, accumulate_params=True, bf="bf16", seed=10)
    colsum_case(ops, 256, 151296, torch.float32, seed=11)


# ---------------------------------------------------------------------------------------- rejection
def test_rejections_leave_the_library_usable():
    """Misaligned float4 pointers (4 bytes off; leading dimensions still multiples of 4), cols outside the
    supported set and an unknown colsum dtype are refused with HBA_ERR_ARG before any launch; outputs stay as
    they were and valid calls afterwards are still right."""
    ops = _ops()
    from hba import _lib
    cols, rows = 256, 1100
    big = torch.randn(rows + 1, cols + 8, device=DEV)
    x, xm = big[:rows, :cols], big[:rows, 1:cols + 1]                     # aligned / 4 bytes off
    gv = torch.randn(cols + 8, device=DEV)
    g, gm = gv[:cols], gv[1:cols + 1]
    out = torch.full((rows, cols + 8), 7.0, device=DEV)
    y, ym = out[:, :cols], out[:, 1:cols + 1]
    dgb = torch.full((2 * cols + 8,), 7.0, device=DEV)
    ws = torch.empty(2 * 148 * 3 * 1024 + 2 * rows + 256 * cols, device=DEV)
    opb = torch.full((rows, 2 * cols + 16), 7.0, dtype=torch.bfloat16, device=DEV)
    op_m = ops.Operand(opb[:, 2:], rows, cols, 0)                         # 4-byte but not 8-byte aligned
    conv = torch.randn(2 * 4 + 1, cols + 8, device=DEV)
    tok = torch.zeros(2, 3, dtype=torch.int64, device=DEV)
    LN = ops.layernorm_fwd
    bad = [
        (lambda: LN(xm, rows, cols, g, g, 1e-5, y_f32=y), "16-byte"),             # streaming form (>= 1024 rows)
        (lambda: LN(xm, 100, cols, g, g, 1e-5, y_f32=y), "16-byte"),              # per-row form
        (lambda: LN(x, 100, cols, gm, g, 1e-5, y_f32=y), "16-byte"),
        (lambda: LN(x, 100, cols, g, gm, 1e-5, y_f32=y), "16-byte"),
        (lambda: LN(x, 100, cols, g, g, 1e-5, y_f32=ym), "16-byte"),
        (lambda: LN(big[:, :100], 100, 100, g, g, 1e-5, y_f32=y), "multiple of 128"),
        (lambda: LN(big.new_empty(10, 1160), 10, 1152, g.new_empty(1152), g.new_empty(1152), 1e-5,
                    y_f32=big.new_empty(10, 1152)), "multiple of 128"),
        (lambda: ops.layernorm_bwd(xm, x, 100, cols, g, 1e-5, y), "16-byte"),
        (lambda: ops.layernorm_bwd(x, xm, 100, cols, g, 1e-5, y), "16-byte"),
        (lambda: ops.layernorm_bwd(x, x, 100, cols, gm, 1e-5, y), "16-byte"),
        (lambda: ops.layernorm_bwd(x, x, 100, cols, g, 1e-5, ym), "16-byte"),
        (lambda: ops.layernorm_bwd(big[:, :100], big[:, :100], 100, 100, g, 1e-5, y), "multiple of 128"),
        (lambda: ops.layernorm_bwd_fused(xm, x, 100, cols, g, 1e-6, y, dgb, ws), "16-byte"),
        (lambda: ops.layernorm_bwd_fused(x, xm, 100, cols, g, 1e-6, y, dgb, ws), "16-byte"),
        (lambda: ops.layernorm_bwd_fused(x, x, 100, cols, gm, 1e-6, y, dgb, ws), "16-byte"),
        (lambda: ops.layernorm_bwd_fused(x, x, 100, cols, g, 1e-6, ym, dgb, ws), "16-byte"),
        (lambda: ops.layernorm_bwd_fused(x, x, 100, cols, g, 1e-6, y, dgb, ws, dx_op=op_m), "8-byte"),
        (lambda: ops.layernorm_bwd_fused(big[:, :384], big[:, :384], 10, 384, gv.new_empty(384), 1e-6,
                                         big.new_empty(10, 384), dgb.new_empty(768), ws), "cols=384"),
        (lambda: ops.layernorm_param_grad(x, xm, 100, cols, 1e-6, dgb, ws), "16-byte"),
        (lambda: ops.layernorm_param_grad(x, big.view(-1)[:100 * (cols + 1)].view(100, cols + 1)[:, :cols], 100, cols,
                                          1e-6, dgb, ws), "ldx"),
        (lambda: ops.assemble_tokens_ln(conv[1:, 1:cols + 1], 2, 4, cols, g, conv[:5, :cols], g, g, 1e-5, y), "16-byte"),
        (lambda: ops.assemble_tokens_ln(conv[:8, :cols], 2, 4, cols, gm, conv[:5, :cols], g, g, 1e-5, y), "16-byte"),
        (lambda: ops.assemble_tokens_ln(conv[:8, :cols], 2, 4, cols, g, conv[:5, 1:cols + 1], g, g, 1e-5, y),
         "16-byte"),
        (lambda: ops.assemble_tokens_ln(conv[:8, :cols], 2, 4, cols, g, conv[:5, :cols], gm, g, 1e-5, y), "16-byte"),
        (lambda: ops.assemble_tokens_ln(conv[:8, :cols], 2, 4, cols, g, conv[:5, :cols], g, gm, 1e-5, y), "16-byte"),
        (lambda: ops.assemble_tokens_ln(conv[:8, :cols], 2, 4, cols, g, conv[:5, :cols], g, g, 1e-5, ym), "16-byte"),
        (lambda: ops.embed_tokens(tok, conv[:, 1:cols + 1], conv[:3, :cols], y), "16-byte"),
        (lambda: ops.embed_tokens(tok, conv[:, :cols], conv[:3, 1:cols + 1], y), "16-byte"),
        (lambda: ops.embed_tokens(tok, conv[:, :cols], conv[:3, :cols], ym), "16-byte"),
        (lambda: ops.check(_lib.load().hba_colsum(ops._p(x), 7, 100, cols, x.stride(0), ops._p(dgb), 0, ops._p(ws),
                                                  ops._stream()), "hba_colsum"), "dtype"),
    ]
    for i, (fn, msg) in enumerate(bad):
        before, before_d, before_b = out.clone(), dgb.clone(), opb.clone()
        with pytest.raises(RuntimeError, match=rf"code {HBA_ERR_ARG}\).*{msg}"):
            fn()
        _sync()
        assert torch.equal(out, before) and torch.equal(dgb, before_d) and torch.equal(opb, before_b), \
            (i, msg, "a rejected call wrote its output")
    # valid calls afterwards: the library is still usable and right
    ln_fwd_case(ops, 1025, 768, outs=("f32", "hilo"), seed=21)
    ln_bwd_case(ops, 9, 256, accumulate=True, seed=22)
    bwd_fused_case(ops, 100, 512, bf="hilo", seed=23)
    colsum_case(ops, 300, 100, torch.bfloat16, seed=24)
