"""hba_gemm_bf16 at every tile, tail and epilogue branch of its launcher, against the fp64 reference of
tests/gemm_ref.py, element by element.

Every output element is checked as |C - ref| <= bound, where (tests/gemm_ref.py: tau(), bound(), sfu_error())
  bound = slope * (tau * S + 2u (|alpha acc| + |bias|)) + sfu + 2u |C| + u |residual| + r_out (|C| + ...)
  S     = |alpha| (|A_hi| + |A_lo|) . (|B_hi| + |B_lo|)^T, per element, in fp64
  tau   = 2^-23 (nsplit K + slices): a bf16 x bf16 product is exact in fp32, so the only GEMM error is the
          accumulation of nsplit * K products (plus the split-K reduction of `slices` partial sums) in fp32;
          each addition loses at most one ulp (2^-23) of a running sum whose magnitude S bounds.  That is the
          worst case of a truncating accumulator; in fp32 mode the reference product is hi.hi + lo.hi + hi.lo,
          so the dropped lo.lo term (<= 2^-16 S) is not an error of the kernel.
  slope = |act'(z)| for QuickGELU / GELU, |act'(aux)| for the gradients, 1 otherwise
  sfu   = the stated accuracy of the activation code at an exact argument: 2-ulp ex2 / rcp / fdividef for
          QuickGELU, 1.5e-7 in erf (Abramowitz-Stegun 7.1.26) plus the SFU roundings for GELU
  u     = 2^-24: one rounding each for alpha * acc, + bias, the activation product and + residual
  r_out = one rounding of the stored type: 0 for f32, 2^-8 for bf16 hi (8 significant bits, round to nearest),
          2^-16 for bf16 hi + lo (lo is the rounded remainder).
The bound is an a-priori worst case, not fitted: random-sign accumulation errors grow like sqrt(K) while the bound
grows like K, so the worst observed |C - ref| / bound sits one to three orders of magnitude below 1 (printed at the
end of the module, by path).  Sensitivity comes from the inputs, not from a tight tolerance: rows of A and
columns of B are scaled over 2^-10 .. 2^10 (a max |C|-normalised error cannot hide a small-magnitude tile), and
dominant products sit at the edges of warps, tiles, k-blocks and split-K slices, so that a dropped or doubled
k-block, pass, row or column moves its element by far more than its bound.

Also: canaries around every output (padded leading dimensions, NaN borders), NaN in the operand padding, bit-exact
invariance under max_ctas / row slicing / repeated launches (which covers tail splitting: a split schedule gives
the bits of the unsplit one), the production shapes of both trainers and argument rejection."""
import contextlib
import itertools
import os
import sys

import pytest
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from gemm_ref import (GELU, GELU_GRAD, GRAD_ACTS, NONE, QUICKGELU, QUICKGELU_GRAD, U32,  # noqa: E402
                      bound, branches, reference, scaled_inputs, spike_plan, split_hi_lo, tau)

pytestmark = pytest.mark.gpu

DEV = "cuda"
HBA_ERR_ARG = -22
NAN = float("nan")
ACT_NAMES = {NONE: "none", QUICKGELU: "quickgelu", GELU: "gelu", QUICKGELU_GRAD: "quickgelu_grad",
             GELU_GRAD: "gelu_grad"}
WORST = {}   # path -> worst |C - ref| / bound over the module (printed at its end)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst |C - ref| / bound by path (tolerance 1):")
        for k in sorted(WORST):
            print(f"  {k:40s} {WORST[k]:.3e}")


def _ops():
    import hba  # noqa: F401
    from hba import ops
    return ops


def _c8(n):
    return (n + 7) // 8 * 8


def _c4(n):
    return (n + 3) // 4 * 4


def _c64(n):
    return (n + 63) // 64 * 64


# ---------------------------------------------------------------------------------------- buffers
class Canvas:
    """Every buffer a call writes, each a padded allocation filled with NaN (bf16: the NaN bit pattern 0x7fc0)
    of which only `regions` (row count, [(first column, width)]) is the logical output; `untouched()` asserts that
    no byte outside those regions changed."""

    def __init__(self):
        self.bufs = []

    def __call__(self, rows, ld, dtype, regions, extra_rows=1):
        buf = torch.full((rows + extra_rows, ld), NAN, dtype=dtype, device=DEV)
        self.bufs.append((buf, rows, regions, buf.clone()))
        return buf

    def untouched(self, what=""):
        for buf, rows, regions, init in self.bufs:
            mask = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
            for c0, w in regions:
                mask[:rows, c0:c0 + w] = False
            bits = (lambda t: t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32))
            assert torch.equal(bits(buf)[mask], bits(init)[mask]), f"{what}: write outside the logical output"


def _operand(ops, x32, nsplit, mn, fill=NAN, zero_pad_hi=True):
    """The operand of logical value x32 [R, K] as the kernel reads it: K-major [R + 1, ld] (hi at [0, K), zero
    up to ceil64(K) in fp32 mode as documented, lo at [lo_off, lo_off + K)) or MN-major [K + 1, ld] (hi at [0, R),
    lo at [lo_off, lo_off + R)), everything else `fill`.  Returns (Operand, hi view, lo view or None)."""
    R, K = x32.shape
    hi, lo = split_hi_lo(x32.to(DEV)) if nsplit == 3 else (x32.to(DEV).to(torch.bfloat16), None)
    if mn:
        hi, lo = hi.t(), (lo.t() if lo is not None else None)
        rows, width = K, R
    else:
        rows, width = R, K
    lo_off = (_c8(width) + 8 if mn else _c64(K) + 16) if nsplit == 3 else 0
    ld = (lo_off if nsplit == 3 else _c8(width)) + _c8(width) + 8
    buf = torch.full((rows + 1, ld), fill, dtype=torch.bfloat16, device=DEV)
    buf[:rows, :width] = hi
    if nsplit == 3:
        if not mn and zero_pad_hi:
            buf[:rows, K:_c64(K)] = 0
        buf[:rows, lo_off:lo_off + width] = lo
    op = ops.Operand(buf, rows, width, lo_off)
    return op, buf[:rows, :width], (buf[:rows, lo_off:lo_off + width] if nsplit == 3 else None)


def _input_f32(x, ld, fill=NAN):
    """x [rows, cols] fp32 or bf16 in a [rows + 1, ld] buffer whose padding holds `fill`."""
    buf = torch.full((x.shape[0] + 1, ld), fill, dtype=x.dtype, device=DEV)
    buf[:x.shape[0], :x.shape[1]] = x.to(DEV)
    return buf[:x.shape[0], :x.shape[1]]


def _record(path, got, ref_val, bnd, what):
    d = (got.double() - ref_val).abs()
    ratio = torch.where(bnd > 0, d / bnd.clamp_min(1e-300), torch.where(d == 0, 0.0, float("inf")))
    ratio = torch.where(torch.isnan(d), float("inf"), ratio)
    worst = float(ratio.max()) if ratio.numel() else 0.0
    WORST[path] = max(WORST.get(path, 0.0), worst)
    if not worst <= 1.0:
        idx = int(ratio.flatten().argmax())
        r, c = divmod(idx, ratio.shape[1])
        raise AssertionError(f"{what} {path}: |C - ref| / bound = {worst:.3g} at [{r}, {c}]: got "
                             f"{float(got.flatten()[idx])!r}, ref {float(ref_val.flatten()[idx])!r}, "
                             f"bound {float(bnd.flatten()[idx]):.3g}")


# ---------------------------------------------------------------------------------------- one checked call
def gemm_case(ops, M, N, K, *, nsplit=1, a_mn=False, b_mn=False, act=NONE, bias=False, residual=False, alpha=1.0,
              pre=None, outs=("f32",), transpose=False, aux=None, aux_ld4=True, k_slices=1, max_ctas=0, seed=0,
              span=None, spikes=None, fill=NAN, zero_pad_hi=True, rows=None, check=True, inputs=None):
    """Builds seeded inputs (scaled rows / columns, dominant products from spike_plan), runs one hba_gemm_bf16
    call with every output inside a NaN canvas, checks the canvas, checks every output against the fp64
    reference element by element, and returns {output name: tensor} for bit comparisons.
    pre: None / "f32" / "bf16"; outs: "f32", "bf16" (hi only), "hilo", "colsum"; aux: None / "f32" / "bf16";
    rows = (r0, m): run on rows [r0, r0 + m) of the M-row problem through narrowed views (no check)."""
    if span is None:
        span = 10 if act == NONE else 2
    if spikes is None:
        spikes = spike_plan(M, N, K)
    a32, b32 = scaled_inputs(M, N, K, seed=seed, spikes=spikes, span=span) if inputs is None else inputs
    g = torch.Generator().manual_seed(seed + 1)
    A, a_hi, a_lo = _operand(ops, a32, nsplit, a_mn, fill, zero_pad_hi)
    B, b_hi, b_lo = _operand(ops, b32, nsplit, b_mn, fill, zero_pad_hi)
    scale = a32.abs().mean(1, keepdim=True) * b32.abs().mean(1) * K ** 0.5   # ~ |C| per element
    bias_t = _input_f32((torch.randn(1, N, generator=g) * 2.0), _c4(N) + 4)[0] if bias else None
    res_t = _input_f32(torch.randn(M, N, generator=g) * scale, _c4(N) + 4) if residual else None
    aux_t = None
    if act in GRAD_ACTS:
        aux_t = _input_f32((torch.randn(M, N, generator=g) * 2.5).to(torch.float32 if aux == "f32" else torch.bfloat16),
                           _c4(N) + (4 if aux_ld4 else 1))
    m0, Mr = (0, M) if rows is None else rows
    if rows is not None:   # narrowed views of the same storage
        assert not a_mn
        A = ops.Operand(A.buf[m0:], Mr, A.K, A.lo_off)
        a_hi, a_lo = a_hi[m0:m0 + Mr], (a_lo[m0:m0 + Mr] if a_lo is not None else None)
        res_t = res_t[m0:m0 + Mr] if res_t is not None else None
        aux_t = aux_t[m0:m0 + Mr] if aux_t is not None else None
    cv = Canvas()
    o = {}
    R, Cn = (N, Mr) if transpose else (Mr, N)    # stored layout of the outputs
    if "f32" in outs:
        o["f32"] = cv(R, _c4(Cn) + 4, torch.float32, [(0, Cn)])
    bf = "hilo" if "hilo" in outs else ("bf16" if "bf16" in outs else None)
    lo_off = 0
    if bf:
        lo_off = _c8(Cn) + 8 if bf == "hilo" else 0
        o[bf] = cv(R, lo_off + _c8(Cn) + 8, torch.bfloat16, [(0, Cn)] + ([(lo_off, Cn)] if lo_off else []))
    if pre:
        o["pre"] = cv(Mr, _c8(N) + 8, torch.float32 if pre == "f32" else torch.bfloat16, [(0, N)])
    groups = (Mr + 31) // 32
    if "colsum" in outs:
        o["colsum"] = cv(1, (groups + 1) * N, torch.float32, [(0, groups * N)], extra_rows=0)
    ws = torch.full((k_slices * Mr * N,), NAN, device=DEV) if k_slices > 1 else None
    ops.gemm(A, B, Mr, K=K, a_mn=a_mn, b_mn=b_mn, act=act, alpha=alpha, bias=bias_t, residual=res_t, aux=aux_t,
             pre_out=o["pre"][:Mr, :N] if pre else None,
             out_f32=o["f32"][:R, :Cn] if "f32" in outs else None,
             out=ops.Operand(o[bf][:R], R, Cn, lo_off) if bf else None,
             colsum_partial=o["colsum"][0] if "colsum" in outs else None,
             transpose_out=transpose, max_ctas=max_ctas, k_slices=k_slices, k_workspace=ws)
    torch.cuda.synchronize()
    what = f"M={M} N={N} K={K} nsplit={nsplit} a_mn={a_mn} b_mn={b_mn} act={act} k_slices={k_slices} " \
           f"max_ctas={max_ctas} rows={rows}"
    cv.untouched(what)
    got = {k: (v[:R, :Cn] if k in ("f32",) else v) for k, v in o.items()}
    if bf:
        hi = o[bf][:R, :Cn]
        got[bf] = hi.float() + (o[bf][:R, lo_off:lo_off + Cn].float() if lo_off else 0)
        got[bf + ".hi_bits"] = hi
    if pre:
        got["pre"] = o["pre"][:Mr, :N]
    if "colsum" in outs:
        got["colsum"] = o["colsum"][0, :groups * N].view(groups, N)
    if not check:
        return got
    ref = reference(a_hi, b_hi, a_lo, b_lo, a_mn=a_mn, b_mn=b_mn, K=K, alpha=alpha, bias=bias_t, act=act,
                    aux=aux_t, residual=res_t)
    t = tau(K, nsplit, branches(Mr, N, K, nsplit, a_mn, b_mn, k_slices)["slices"])
    path = f"nsplit{nsplit}.{ACT_NAMES[act]}"
    for k in ("f32", "bf16", "hilo"):
        if k not in got:
            continue
        v = got[k].t() if transpose else got[k]
        bnd = bound(ref, t, act, k, bias=bias_t, residual=res_t, alpha=alpha)
        _record(f"{path}.{'T.' if transpose else ''}{k}", v, ref["C"], bnd, what)
    if pre:
        _record(f"{path}.pre_{pre}", got["pre"], ref["z"],
                bound(ref, t, act, pre, bias=bias_t, alpha=alpha, pre=True), what)
    if "colsum" in outs:
        # the kernel's own bf16 hi outputs, summed per 32-row group: at most 31 fp32 additions
        hi = got[bf + ".hi_bits"].double()
        pad = torch.zeros(groups * 32 - Mr, N, dtype=torch.float64, device=hi.device)
        h = torch.cat([hi, pad]).view(groups, 32, N)
        _record(f"{path}.colsum", got["colsum"], h.sum(1), 31 * U32 * h.abs().sum(1), what)
    if "f32" in got and bf == "bf16" and not transpose:   # the bf16 output is the rounded fp32 one
        assert torch.equal(got["bf16.hi_bits"], got["f32"].to(torch.bfloat16)), what
    return got


# ---------------------------------------------------------------------------------------- sweep
SWEEP_M = [256, 100, 128, 200, 192]          # M tail: none, peer CTA empty (M % 32 != 0 / == 0), peer partial (both)
SWEEP_N = [128, 176, 132, 131, 512, 304, 276, 259]   # BN = 128 / 256: full, N % 16 == 0, N % 4 == 0, ragged
SWEEP_K = [448, 450, 64, 40]                 # k-blocks >= stages or not, ragged last k-block or not
MAJORS = list(itertools.product([False, True], [False, True]))


@pytest.mark.parametrize("a_mn,b_mn", MAJORS)
@pytest.mark.parametrize("nsplit", [1, 3])
@pytest.mark.parametrize("M,N", list(itertools.product(SWEEP_M, SWEEP_N)))
def test_sweep(M, N, nsplit, a_mn, b_mn):
    """The plain product at every (M tail, N tail, ragged K, short K) class, both modes, all operand majors."""
    ops = _ops()
    for K in SWEEP_K:
        gemm_case(ops, M, N, K, nsplit=nsplit, a_mn=a_mn, b_mn=b_mn, seed=M * 7 + N + K)


# ---------------------------------------------------------------------------------------- epilogues
# scheduling form -> (max_ctas, k_slices, K, [(M, N)]): M tail none / peer empty / peer partial (M % 32 != 0)
# crossed with N tail full / N % 16 == 0 / N % 4 == 0 / ragged
SCHEDULES = {
    "single": (0, 1, 200, [768, 720, 700, 701]),     # 3 tiles on 3 CTA pairs
    "rounds": (2, 1, 448, [768, 720, 700, 701]),     # one CTA pair: 3 items, accumulator stages reused
    "tail2": (4, 1, 130, [768, 720, 700, 601]),      # 3 tiles on 2 pairs: the last one in two slabs (601: one past N)
    "tail4": (8, 1, 264, [1280, 1232, 1220, 1029]),  # 5 tiles on 4 pairs: four slabs (1029: three past N)
    "splitk": (0, 3, 428, [768, 720, 700]),          # 7 k-blocks in slices of 3, 3, 1 (N % 4 == 0 only)
}
SCHED_M = [256, 100, 200]


def _recipes():
    """(name, kwargs): every act bare and with bias + residual + alpha; the outputs, pre_out and aux forms rotate."""
    r = []
    outs_cycle = [("f32",), ("f32", "bf16", "colsum"), ("hilo",), ("bf16", "colsum"), ("f32", "hilo", "colsum")]
    pre_cycle = [None, "f32", "bf16"]
    aux_cycle = [("f32", True), ("bf16", False), ("bf16", True), ("f32", False)]
    n = 0
    for act in (NONE, QUICKGELU, GELU, QUICKGELU_GRAD, GELU_GRAD):
        for full in (False, True):
            kw = dict(act=act, outs=outs_cycle[n % 5], pre=pre_cycle[n % 3])
            if full:
                kw.update(bias=True, residual=True, alpha=0.6875)
            if act in GRAD_ACTS:
                kw["aux"], kw["aux_ld4"] = aux_cycle[n % 4]
            r.append((f"{ACT_NAMES[act]}.{'full' if full else 'bare'}", kw))
            n += 1
    r.append(("transposed.alpha_bias", dict(transpose=True, alpha=0.6875, bias=True, outs=("f32", "hilo"))))
    r.append(("transposed.bf16", dict(transpose=True, outs=("bf16",))))
    return r


RECIPES = _recipes()


def _allowed(kw, sched, N):
    """Drops what the launcher rejects: split-K with colsum / transposed output; colsum with N % 4 != 0."""
    kw = dict(kw)
    if sched == "splitk" and kw.get("transpose"):
        return None
    if "colsum" in kw["outs"] and (sched == "splitk" or N % 4):
        kw["outs"] = tuple(o for o in kw["outs"] if o != "colsum")
    return kw


@pytest.mark.parametrize("recipe", [r[0] for r in RECIPES])
@pytest.mark.parametrize("nsplit", [1, 3])
@pytest.mark.parametrize("sched", list(SCHEDULES))
def test_epilogue(sched, nsplit, recipe):
    ops = _ops()
    max_ctas, k_slices, K, ns = SCHEDULES[sched]
    base = dict(RECIPES)[recipe]
    for M, N in itertools.product(SCHED_M, ns):
        kw = _allowed(base, sched, N)
        if kw is None:
            continue
        ks = [0, K - 1, 191, 192, 383, 384] if k_slices > 1 else None   # first / last k of every slice
        gemm_case(ops, M, N, K, nsplit=nsplit, max_ctas=max_ctas, k_slices=k_slices, seed=M + N + nsplit,
                  spikes=spike_plan(M, N, K, ks), **kw)


# ---------------------------------------------------------------------------------------- operand padding
@pytest.mark.parametrize("a_mn,b_mn", MAJORS)
@pytest.mark.parametrize("nsplit", [1, 3])
@pytest.mark.parametrize("M,N,K", [(200, 259, 130), (300, 176, 450)])
def test_operand_padding_is_not_read(M, N, K, nsplit, a_mn, b_mn):
    """NaN in every byte of the operand buffers outside the problem (columns >= K of a K-major operand, columns
    >= M / N of an MN-major one, the trailing row; in fp32 mode also [ceil64(K), lo_off) of a K-major operand - only
    the documented zero padding of its hi part up to ceil64(K) stays): C is finite and bit-identical to the
    zero-padded run."""
    ops = _ops()
    kw = dict(nsplit=nsplit, a_mn=a_mn, b_mn=b_mn, act=QUICKGELU, bias=True, residual=True,
              outs=("f32", "hilo"), seed=K)
    clean = gemm_case(ops, M, N, K, fill=0.0, **kw)
    dirty = gemm_case(ops, M, N, K, fill=NAN, **kw)
    assert torch.isfinite(dirty["f32"]).all()
    for k in ("f32", "hilo.hi_bits", "hilo"):
        assert torch.equal(clean[k], dirty[k]), k


def test_fp32_mode_needs_the_zero_padded_hi_part():
    """The documented requirement is real: NaN in [K, ceil64(K)) of a K-major hi part reaches C (so the padding
    test above exercises the region the kernel reads)."""
    ops = _ops()
    got = gemm_case(ops, 128, 128, 100, nsplit=3, fill=NAN, zero_pad_hi=False, check=False)
    assert torch.isnan(got["f32"]).any()


# ---------------------------------------------------------------------------------------- invariance
INV_CASES = [
    dict(act=QUICKGELU, bias=True, residual=True, pre="bf16", outs=("f32", "hilo")),
    dict(act=GELU_GRAD, aux="bf16", outs=("bf16", "colsum")),
    dict(alpha=0.6875, bias=True, outs=("f32", "hilo"), transpose=True),
]


def _bits_equal(x, y, what):
    for k in x:
        assert torch.equal(x[k], y[k]), (what, k)


@pytest.mark.parametrize("nsplit", [1, 3])
@pytest.mark.parametrize("M,N,K", [(1000, 1000, 200), (2600, 2048, 130), (2500, 2560, 130), (700, 701, 96)])
def test_max_ctas_invariance(M, N, K, nsplit):
    """One call, the same bits for max_ctas 0 (74 pairs), 2 (one pair: every tile in turn), 14 (7 pairs) and 146
    (73 pairs); (2600, 2048) has 88 tiles: tail split f = 4 with 74 and 73 pairs, none with 7; (2500, 2560) has
    100 tiles: tail split f = 2 with 74, 7 and 73 pairs, none with one pair."""
    ops = _ops()
    for i, kw in enumerate(INV_CASES):
        kw = _allowed(kw, "", N)
        runs = [gemm_case(ops, M, N, K, nsplit=nsplit, max_ctas=mc, seed=i, check=(mc == 0), **kw)
                for mc in (0, 2, 14, 146)]
        for r in runs[1:]:
            _bits_equal(runs[0], r, (M, N, K, i))
    if N % 4 == 0:
        runs = [gemm_case(ops, 66, N, 8 * K, nsplit=nsplit, act=QUICKGELU, bias=True, residual=True,
                          outs=("f32", "hilo"), k_slices=3, max_ctas=mc, check=(mc == 0)) for mc in (0, 2, 14)]
        for r in runs[1:]:
            _bits_equal(runs[0], r, "split-K")


@pytest.mark.parametrize("nsplit", [1, 3])
def test_row_slices_are_bit_exact(nsplit):
    """Rows [r0, r0 + m) computed through narrowed A, residual, aux and outputs equal those rows of the full
    result, bit for bit (the output bits do not depend on M or on a row's place in its tile)."""
    ops = _ops()
    M, N, K = 600, 520, 200
    for kw in (dict(act=QUICKGELU_GRAD, aux="f32", residual=True, bias=True, pre="f32", outs=("f32", "hilo")),
               dict(act=GELU, bias=True, outs=("bf16",), pre="bf16"),
               dict(bias=True, residual=True, outs=("f32",), k_slices=3)):
        full = gemm_case(ops, M, N, K, nsplit=nsplit, seed=5, **kw)
        for r0, m in ((0, 1), (37, 100), (200, 256), (599, 1), (128, 300), (1, 599)):
            part = gemm_case(ops, M, N, K, nsplit=nsplit, seed=5, rows=(r0, m), check=False, **kw)
            for k in part:
                if k != "colsum":
                    assert torch.equal(part[k], full[k][r0:r0 + m]), (kw, r0, m, k)


def test_repeated_launches_and_split_k_are_deterministic():
    ops = _ops()
    for kw in (dict(M=66, N=768, K=3072, k_slices=6, act=QUICKGELU, bias=True, residual=True, pre="bf16",
                    outs=("f32", "hilo")),
               dict(M=1024, N=1024, K=4096, k_slices=8, a_mn=True, b_mn=True, outs=("f32",)),
               dict(M=2600, N=2048, K=130, act=GELU_GRAD, aux="bf16", outs=("bf16", "colsum"))):
        first = gemm_case(ops, nsplit=3 if kw["M"] == 66 else 1, seed=1, **kw)
        for _ in range(2):
            _bits_equal(first, gemm_case(ops, nsplit=3 if kw["M"] == 66 else 1, seed=1, check=False, **kw), kw)


# ---------------------------------------------------------------------------------------- production shapes
# (name, M, N, K, nsplit, gemm_case kwargs) of the calls one training step makes, with their epilogues.
# CLIP ViT-L/14 at batch 32: vision rows 32 x 257 = 8224, width 1024; text rows 66 x 77 = 5082, width 768;
# CLS / EOT rows 32 / 66 through split-K; weight gradients MN-major with auto_k_slices.  ViT-B/16 at the
# benchmark's batch 256: rows 256 x 197 = 50432, width 768; its head with 1000 and 10 classes.
def _prod():
    cases = []
    for tower, M, d in (("vision", 8224, 1024), ("text", 5082, 768)):
        for ns in (1, 3):
            cases += [
                (f"{tower}.qkv", M, 3 * d, d, ns, dict(bias=True, outs=("f32",) if ns == 3 else ("bf16",))),
                (f"{tower}.out_proj", M, d, d, ns, dict(bias=True, residual=True)),
                (f"{tower}.c_fc", M, 4 * d, d, ns, dict(bias=True, act=QUICKGELU, outs=("hilo" if ns == 3 else "bf16",),
                                                        pre="f32" if ns == 3 else "bf16")),
                (f"{tower}.c_proj", M, d, 4 * d, ns, dict(bias=True, residual=True)),
            ]
    for tag, R, d in (("cls", 32, 1024), ("eot", 66, 768)):
        for ns in (1, 3):
            cases += [
                (f"{tag}.out_proj", R, d, d, ns, dict(bias=True, residual=True, k_slices="auto")),
                (f"{tag}.c_fc", R, 4 * d, d, ns, dict(bias=True, act=QUICKGELU, outs=("hilo" if ns == 3 else "bf16",),
                                                      pre="f32" if ns == 3 else "bf16", k_slices="auto")),
                (f"{tag}.c_proj", R, d, 4 * d, ns, dict(bias=True, residual=True, k_slices="auto")),
                (f"{tag}.proj", R, 768, d, ns, dict(k_slices="auto")),
                (f"{tag}.c_proj_dx", R, 4 * d, d, ns, dict(act=QUICKGELU_GRAD, aux="f32" if ns == 3 else "bf16",
                                                           outs=("hilo" if ns == 3 else "bf16",), k_slices="auto")),
                (f"{tag}.c_fc_dx", R, d, 4 * d, ns, dict(k_slices="auto")),
            ]
    for name, Mo, No, R in (("vision.dW_out_proj", 1024, 1024, 8224), ("text.dW_out_proj", 768, 768, 5082),
                            ("cls.dW_c_fc", 4096, 1024, 32), ("vit.dW_fc1", 3072, 768, 50432),
                            ("vit.dW_qkv", 2304, 768, 50432)):
        cases.append((name, Mo, No, R, 1, dict(a_mn=True, b_mn=True, k_slices="auto_w")))
    M = 50432
    cases += [
        ("vit.qkv", M, 2304, 768, 1, dict(bias=True, outs=("bf16",))),
        ("vit.proj", M, 768, 768, 1, dict(bias=True, residual=True)),
        ("vit.fc1", M, 3072, 768, 1, dict(bias=True, act=GELU, outs=("bf16",), pre="bf16")),
        ("vit.fc2", M, 768, 3072, 1, dict(bias=True, residual=True)),
        ("vit.fc2_dx", M, 3072, 768, 1, dict(b_mn=True, act=GELU_GRAD, aux="bf16", outs=("bf16", "colsum"))),
        ("vit.fc1_dx", M, 768, 3072, 1, dict(b_mn=True)),
        ("vit.head1000", 256, 1000, 768, 1, dict(bias=True)),
        ("vit.head10", 256, 10, 768, 1, dict(bias=True)),
        ("vit.head10_dx", 256, 768, 10, 1, dict(b_mn=True)),
    ]
    return cases


PRODUCTION = _prod()


@pytest.mark.parametrize("name", [c[0] + f".nsplit{c[4]}" for c in PRODUCTION])
def test_production_shapes(name):
    ops = _ops()
    _n, M, N, K, ns, kw = next(c for c in PRODUCTION if c[0] + f".nsplit{c[4]}" == name)
    kw = dict(kw)
    if kw.get("k_slices") == "auto":
        kw["k_slices"] = ops.auto_k_slices(M, N, K, min_kblocks=4)
    elif kw.get("k_slices") == "auto_w":
        kw["k_slices"] = ops.auto_k_slices(M, N, K)
    first = gemm_case(ops, M, N, K, nsplit=ns, seed=M + N + K, **kw)
    _bits_equal(first, gemm_case(ops, M, N, K, nsplit=ns, seed=M + N + K, check=False, **kw), name)


# ---------------------------------------------------------------------------------------- rejection
@contextlib.contextmanager
def _patched_params(ops, mutate):
    """Calls made through ops.gemm in this context reach hba_gemm_bf16 with `mutate(params)` applied: argument
    combinations the Python front end refuses on its own."""
    real = ops._lib

    class _Lib:
        def __getattr__(self, name):
            fn = getattr(real.load(), name)
            if name != "hba_gemm_bf16":
                return fn

            def call(pref, stream):
                mutate(pref._obj)
                return fn(pref, stream)
            return call

    class _Shim:
        def __getattr__(self, name):
            return getattr(real, name)

        @staticmethod
        def load():
            return _Lib()

    ops._lib = _Shim()
    try:
        yield
    finally:
        ops._lib = real


def test_rejections_leave_the_library_usable():
    ops = _ops()
    M, N, K = 200, 260, 128
    a = ops.Operand(torch.randn(M, K, device=DEV).to(torch.bfloat16), M, K, 0)
    b = ops.Operand(torch.randn(N, K, device=DEV).to(torch.bfloat16), N, K, 0)
    out = torch.full((M, N), 777.0, device=DEV)
    pre = torch.randn(M, N + 4, device=DEV)
    preb = torch.randn(M, N + 4, device=DEV).to(torch.bfloat16)
    ws = torch.empty(3 * M * N, device=DEV)
    a3 = ops.Operand.empty(M, K, True, DEV, zero=True)
    b3 = ops.Operand.empty(N, K, True, DEV, zero=True)
    bad = [
        # aux read as float4 / 8-byte vectors (ld % 4 == 0) from a view that is only 4- / 2-byte aligned
        (lambda: ops.gemm(a, b, M, act=GELU_GRAD, aux=pre[:, 1:N + 1], out_f32=out), "aux", None),
        (lambda: ops.gemm(a, b, M, act=QUICKGELU_GRAD, aux=preb[:, 2:N + 2], out_f32=out), "aux", None),
        (lambda: ops.gemm(a, ops.Operand(b.buf[:N - 2], N - 2, K, 0), M, out=ops.Operand(
            torch.empty(M, N + 4, dtype=torch.bfloat16, device=DEV), M, N - 2, 0),
            colsum_partial=torch.empty(7 * N, device=DEV)), "colsum_partial", None),
        (lambda: ops.gemm(a, b, M, out_f32=out, k_slices=3, k_workspace=ws), "split-K",
         lambda p: setattr(p, "k_workspace", None)),
        (lambda: ops.gemm(a, b, M, out_f32=out, act=QUICKGELU, transpose_out=True), "transpose_out", None),
        (lambda: ops.gemm(a3, b3, M, out_f32=out), "lo offsets", lambda p: setattr(p, "a_lo_off", 64 - 8)),
    ]
    for fn, msg, mutate in bad:
        before = out.clone()
        with _patched_params(ops, mutate) if mutate else contextlib.nullcontext():
            with pytest.raises(RuntimeError, match=rf"code {HBA_ERR_ARG}\).*{msg}"):
                fn()
        torch.cuda.synchronize()
        assert torch.equal(out, before), (msg, "a rejected call wrote its output")
    # the aligned forms of the same aux views run, and a valid GEMM afterwards is still right
    ops.gemm(a, b, M, act=GELU_GRAD, aux=pre[:, 4:N + 4], out_f32=out)
    ops.gemm(a, b, M, act=QUICKGELU_GRAD, aux=preb[:, 4:N + 4], out_f32=out)
    gemm_case(ops, 200, 701, 130, act=QUICKGELU, bias=True, residual=True, outs=("f32", "hilo"), nsplit=3)

