"""The fp64 references, the error bound, the branch map and the inputs of tests/rowwise_ref.py that
tests/test_gpu_rowwise_shapes.py relies on, checked without a GPU: against torch and fp64 autograd, against an fp32
emulation of the kernels (which must pass) and its mutants (which must fail); and a dry run of the GPU file on the
CPU restatement of libhba."""
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from rowwise_ref import (EPS_CLIP, EPS_TIMM, FUSED_COLS, assemble_x, bwd_dy, bwd_fused_branches,  # noqa: E402
                         colsum_branches, colsum_ref, emulate_ln_bwd, emulate_ln_fwd, ln_bwd_bound, ln_bwd_ref,
                         ln_fwd_bound, ln_fwd_branches, ln_fwd_ref, ln_fwd_stages, ln_params, ln_rows, ln_stats,
                         param_grad_ref, strided)
from test_gpu_rowwise_shapes import (CS_SHAPES, FUSED_ROWS, PG_SHAPES, SWEEP_COLS, fwd_rows)  # noqa: E402


@pytest.mark.parametrize("eps", [EPS_CLIP, EPS_TIMM])
@pytest.mark.parametrize("cols", [128, 384, 1024])
def test_reference_matches_torch_and_autograd(cols, eps):
    x = ln_rows(37, cols, seed=cols, eps=eps)
    gamma, beta = ln_params(cols, 1)
    dy = bwd_dy(x, gamma, eps, 2)
    st = ln_fwd_ref(x, gamma, beta, eps)
    xd = x.double().requires_grad_(True)
    gd, bd = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    y = F.layer_norm(xd, (cols,), gd, bd, float(torch.tensor(eps, dtype=torch.float32)))
    torch.testing.assert_close(st["y"], y.detach(), rtol=1e-12, atol=1e-10)
    y.backward(dy.double())
    prev = torch.randn(37, cols, dtype=torch.float64)
    b = ln_bwd_ref(dy, x, gamma, eps, prev)
    torch.testing.assert_close(b["dx"], xd.grad + prev, rtol=1e-9, atol=1e-9)
    p = param_grad_ref(dy, x, eps)
    torch.testing.assert_close(p["dgamma"], gd.grad, rtol=1e-9, atol=1e-9)
    torch.testing.assert_close(p["dbeta"], bd.grad, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(colsum_ref(dy), dy.double().sum(0), rtol=1e-15, atol=0)
    xb = dy.to(torch.bfloat16)
    torch.testing.assert_close(colsum_ref(xb), xb.double().sum(0), rtol=1e-15, atol=0)


def test_assembly_reference():
    g = torch.Generator().manual_seed(0)
    B, n, w = 2, 3, 128
    conv, cls, pos = torch.randn(B * n, w, generator=g), torch.randn(w, generator=g), torch.randn(n + 1, w, generator=g)
    x = assemble_x(conv, cls, pos, B, n).view(B, n + 1, w)
    assert torch.equal(x[1, 0], cls + pos[0]) and torch.equal(x[1, 2], conv[n + 1] + pos[2])
    gamma, beta = ln_params(w, 0)
    st = ln_fwd_ref(x.view(-1, w), gamma, beta, EPS_CLIP)
    torch.testing.assert_close(st["y"], F.layer_norm(x.view(-1, w).double(), (w,), gamma.double(), beta.double(),
                                                     float(torch.tensor(EPS_CLIP, dtype=torch.float32))))


def test_inputs_have_the_advertised_rows():
    x = ln_rows(60, 256, seed=0, eps=EPS_CLIP)
    st = ln_stats(x, EPS_CLIP)
    ratio = (st["mean"].abs() / st["var"].sqrt().clamp_min(1e-30)).squeeze(1)
    assert float(ratio[1::6].max()) > 2 ** 9                               # offset rows up to 2^10
    assert float(st["var"][2::6].max()) < EPS_CLIP * 2 ** -10              # var << eps
    assert float(st["var"][3::6].abs().max()) == 0 and float(st["mean"][3::6].abs().min()) > 0    # constant rows
    assert float(x[5::6].abs().max()) == 0
    gamma, beta = ln_params(256, 0)
    assert (gamma == 0).sum() > 30 and (gamma < 0).any() and (gamma > 0).any() and float(beta.abs().mean()) > 8
    # dy of the null-space rows: g is (a + b xhat) up to 2^-10 noise, so dx << |g| r
    gamma, _ = ln_params(256, 0, zeros=False)
    dy = bwd_dy(x, gamma, EPS_CLIP, 0)
    b = ln_bwd_ref(dy, x, gamma, EPS_CLIP)
    null = [r for r in range(0, 60, 3) if float(b["var"][r]) > 1e-3]
    assert float((b["z"][null].abs().amax(1) / b["g"][null].abs().amax(1)).max()) < 1e-2


# ---------------------------------------------------------------------------------------- branch map
def test_branch_map_hand_cases():
    assert [ln_fwd_stages(c) for c in SWEEP_COLS] == [8, 8, 6, 4, 3, 2, 2, 2]
    assert ln_fwd_branches(1023, 768)["form"] == "per_row"
    b = ln_fwd_branches(1024, 768)
    assert (b["form"], b["grid"], b["rows_min"], b["rows_max"], b["partial_last"]) == ("stream", 43, 23, 24, True)
    b = ln_fwd_branches(3552, 128)
    assert (b["grid"], b["iters_max"], b["partial_last"], b["wraps"]) == (148, 1, False, 0)
    b = ln_fwd_branches(3553, 128)
    assert (b["grid"], b["iters_max"], b["rows_max"], b["partial_last"]) == (148, 2, 25, True)
    assert ln_fwd_branches(3528, 128)["grid"] == 147 and ln_fwd_branches(3529, 128)["grid"] == 148
    b = ln_fwd_branches(8224, 1024)                      # CLIP-HBA vision rows: 55 or 56 rows, 3 iterations, 1 wrap
    assert (b["grid"], b["rows_min"], b["rows_max"], b["iters_max"], b["wraps"]) == (148, 55, 56, 3, 1)
    b = bwd_fused_branches(50432, 768)
    assert (b["nvec"], b["blocks"], b["rows_per_warp_max"], b["rows_per_warp_min"]) == (6, 296, 22, 21)
    assert bwd_fused_branches(9, 128)["blocks"] == 2 and bwd_fused_branches(2368, 128)["rows_per_warp_max"] == 1
    assert colsum_branches(1, 33) == {"per": 1, "empty_chunks": 127, "col_blocks": 2, "partial_col_block": True}
    assert colsum_branches(129, 64)["empty_chunks"] == 63 and colsum_branches(256, 64)["empty_chunks"] == 0


def test_sweep_reaches_every_branch_combination():
    """The GPU sweep reaches every stages value, a grid below 148 and of 148, one and several ring wraps, a partial
    last stage (with and without wraps), every NVEC, one and several rows per warp, empty chunks and partial column
    blocks."""
    stages, seen = set(), set()
    for cols in SWEEP_COLS:
        for rows in fwd_rows(cols):
            b = ln_fwd_branches(rows, cols)
            seen.add(("form", b["form"]))
            if b["form"] == "stream":
                stages.add(b["stages"])
                seen |= {("grid148", b["grid"] == 148), ("partial", b["partial_last"])}
                seen.add(("wraps", min(b["wraps"], 2), b["stages"]))
    assert stages == {8, 6, 4, 3, 2}
    assert {("grid148", False), ("grid148", True), ("partial", True), ("partial", False)} <= seen
    for s in stages:
        assert {("wraps", 0, s), ("wraps", 1, s), ("wraps", 2, s)} <= seen, s
    assert {bwd_fused_branches(r, c)["nvec"] for c in FUSED_COLS for r in FUSED_ROWS} == {1, 2, 4, 6, 8}
    per_warp = {bwd_fused_branches(r, 128)["rows_per_warp_max"] > 1 for r in FUSED_ROWS}
    assert per_warp == {False, True}
    cs = {(colsum_branches(r, c)["empty_chunks"] > 0, colsum_branches(r, c)["partial_col_block"])
          for r, c in PG_SHAPES + CS_SHAPES}
    assert cs == {(False, False), (False, True), (True, False), (True, True)}


# ---------------------------------------------------------------------------------------- the bound catches defects
def _ok(got, ref, bnd):
    return bool(((got.double() - ref).abs() <= bnd).all())


@pytest.mark.parametrize("cols", [128, 1024])
@pytest.mark.parametrize("eps", [EPS_CLIP, EPS_TIMM])
def test_bound_catches_what_the_kernel_could_get_wrong(cols, eps):
    """A faithful fp32 emulation of the kernels passes the bound; unbiased variance, eps outside the square root, a
    float4 chunk left out of the statistics, row_step applied to dy, accumulation into the wrong row and the partial
    last stage of a streaming CTA dropped each fail on the generated inputs."""
    rows, step = 1025, 3
    x = ln_rows(rows, cols, seed=cols, eps=eps)
    gamma, beta = ln_params(cols, 2)
    st = ln_fwd_ref(x, gamma, beta, eps)
    bnd = ln_fwd_bound(st)
    assert _ok(emulate_ln_fwd(x, gamma, beta, eps), st["y"], bnd)
    for m in ("unbiased", "eps_outside", "skip_chunk", "drop_last_stage"):
        assert not _ok(emulate_ln_fwd(x, gamma, beta, eps, mutant=m), st["y"], bnd), m
    gamma, _ = ln_params(cols, 2, zeros=False)
    dy = bwd_dy(x, gamma, eps, 3)
    dy_all = strided(dy, step, 3)                           # dy rows r (the kernel), r * step (the mutant)
    dy_all[:rows] = dy
    prev = torch.randn(rows, cols, generator=torch.Generator().manual_seed(4)) * 4
    b = ln_bwd_ref(dy, x, gamma, eps, prev)
    bb = ln_bwd_bound(b)
    assert _ok(emulate_ln_bwd(dy_all, x, gamma, eps, prev, step), b["dx"], bb)
    for m in ("dy_row_step", "wrong_row", "unbiased", "eps_outside", "skip_chunk"):
        assert not _ok(emulate_ln_bwd(dy_all, x, gamma, eps, prev, step, mutant=m), b["dx"], bb), m
    bp = ln_bwd_ref(dy, x, gamma, eps)
    assert _ok(emulate_ln_bwd(dy_all, x, gamma, eps, None, step), bp["dx"], ln_bwd_bound(bp))


# ---------------------------------------------------------------------------------------- dry run
def test_gpu_test_file_dry_runs_on_the_cpu_restatement():
    """tests/test_gpu_rowwise_shapes.py itself, run by pytest on the CPU with libhba served by its restatement; left
    out: the production shapes (fp64 references of 50432 x 768 and 256 x 151296 are minutes of CPU time)."""
    tool = os.path.join(ROOT, "tests", "emulate_clip_gpu_tests.py")
    out = subprocess.run([sys.executable, tool, os.path.join(ROOT, "tests", "test_gpu_rowwise_shapes.py"), "-k",
                          "not production"],
                         capture_output=True, text=True, timeout=3000, env=dict(os.environ, OMP_NUM_THREADS="8"))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    tail = [line for line in out.stdout.splitlines() if " passed" in line][-1]
    assert "failed" not in tail and "error" not in tail and int(tail.split(" passed")[0].split()[-1]) >= 76, tail
