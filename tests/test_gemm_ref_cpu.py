"""The fp64 GEMM reference, the launcher's branch map and the scaled / spiked inputs that
tests/test_gpu_gemm_shapes.py relies on, checked without a GPU; and a dry run of that file on the CPU
restatement of libhba."""
import itertools
import os
import subprocess
import sys

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from gemm_ref import (GELU, GELU_GRAD, NONE, QUICKGELU, QUICKGELU_GRAD, bound, branches,  # noqa: E402
                      n_class, reference, scaled_inputs, spike_plan, split_hi_lo, tau)
from test_gpu_gemm_shapes import MAJORS, SCHED_M, SCHEDULES, SWEEP_K, SWEEP_M, SWEEP_N  # noqa: E402

ACTS = (NONE, QUICKGELU, GELU, QUICKGELU_GRAD, GELU_GRAD)


def _autograd_act(act, x):
    """act' by autograd of torch's own activation (QuickGELU as CLIP writes it, exact erf-GELU)."""
    x = x.clone().requires_grad_(True)
    y = x * torch.sigmoid(1.702 * x) if act == QUICKGELU_GRAD else F.gelu(x)
    y.backward(torch.ones_like(y))
    return x.grad


@pytest.mark.parametrize("act", ACTS)
@pytest.mark.parametrize("a_mn,b_mn", MAJORS)
def test_reference_matches_torch(act, a_mn, b_mn):
    g = torch.Generator().manual_seed(act * 4 + 2 * a_mn + b_mn)
    M, N, K = 37, 29, 70
    a = torch.randn(M, K, generator=g, dtype=torch.float64)
    b = torch.randn(N, K, generator=g, dtype=torch.float64)
    bias, res = torch.randn(N, generator=g, dtype=torch.float64), torch.randn(M, N, generator=g, dtype=torch.float64)
    aux = torch.randn(M, N, generator=g, dtype=torch.float64) * 3
    # operands in their stored layout, with columns (K-major) or rows (MN-major) past K it must ignore
    sa = torch.cat([a, torch.full((M, 5), float("nan"), dtype=torch.float64)], 1) if not a_mn else \
        torch.cat([a.t(), torch.full((5, M), float("nan"), dtype=torch.float64)], 0)
    sb = torch.cat([b, torch.full((N, 5), float("nan"), dtype=torch.float64)], 1) if not b_mn else \
        torch.cat([b.t(), torch.full((5, N), float("nan"), dtype=torch.float64)], 0)
    r = reference(sa, sb, a_mn=a_mn, b_mn=b_mn, K=K, alpha=0.75, bias=bias, act=act, aux=aux, residual=res)
    z = 0.75 * F.linear(a, b) + bias
    torch.testing.assert_close(r["z"], z, rtol=1e-12, atol=1e-12)
    if act == NONE:
        want = z
    elif act == QUICKGELU:
        want = z * torch.sigmoid(1.702 * z)
    elif act == GELU:
        want = F.gelu(z)
    else:
        want = z * _autograd_act(act, aux)
    torch.testing.assert_close(r["C"], want + res, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(r["S"], 0.75 * a.abs() @ b.abs().t(), rtol=1e-12, atol=0)


def test_fp32_mode_product_drops_lo_lo():
    """hi.hi + lo.hi + hi.lo: within |lo| . |lo|^T of the unsplit product, which is ~2^-16 of S."""
    g = torch.Generator().manual_seed(3)
    a, b = torch.randn(64, 200, generator=g), torch.randn(48, 200, generator=g)
    (ah, al), (bh, bl) = split_hi_lo(a), split_hi_lo(b)
    r = reference(ah, bh, al, bl)
    hh, ll = ah.double() @ bh.double().t(), al.double() @ bl.double().t()
    torch.testing.assert_close(r["acc"], r["full"] - ll, rtol=1e-13, atol=1e-13)
    assert ((r["acc"] - r["full"]).abs() <= r["lolo"] * (1 + 1e-12)).all()
    assert float((r["lolo"] / r["S"]).max()) < 2.0 ** -15
    # and the unsplit product is the product of the fp32 values to within bf16x2 representation error
    assert float(((r["full"] - a.double() @ b.double().t()).abs() / r["S"]).max()) < 2.0 ** -15
    assert not torch.equal(r["acc"], hh)


@pytest.mark.parametrize("act", ACTS)
def test_reference_matches_the_cpu_restatement(act):
    """oracle/libhba_ref.py (the CPU restatement the dry run serves the GPU file with) computes the same epilogue,
    in fp32: within the same bound the CUDA kernel is held to."""
    from oracle.libhba_ref import emulated_device
    sys.path.insert(0, os.path.join(ROOT, "vit-project_b200"))
    with emulated_device():
        from hba import ops
        M, N, K = 70, 92, 136
        for nsplit in (1, 3):
            a32, b32 = scaled_inputs(M, N, K, seed=act, spikes=spike_plan(M, N, K), span=2)
            g = torch.Generator().manual_seed(act)
            bias, res = torch.randn(N, generator=g), torch.randn(M, N + 4, generator=g)[:, :N]
            aux = torch.randn(M, N + 4, generator=g)[:, :N]
            lo_off = 192 if nsplit == 3 else 0      # fp32 mode: the hi part zero padded up to ceil64(K)
            A, B = (ops.Operand(torch.zeros(x.shape[0], lo_off + 144, dtype=torch.bfloat16), x.shape[0], K, lo_off)
                    for x in (a32, b32))
            for op, x in ((A, a32), (B, b32)):
                hi, lo = split_hi_lo(x)
                op.buf[:, :K] = hi
                if nsplit == 3:
                    op.buf[:, op.lo_off:op.lo_off + K] = lo
            out = torch.empty(M, N + 4)[:, :N]
            ops.gemm(A, B, M, alpha=0.75, bias=bias, act=act, aux=aux if act >= QUICKGELU_GRAD else None,
                     residual=res, out_f32=out)
            lo = (lambda op: op.buf[:, op.lo_off:op.lo_off + K]) if nsplit == 3 else (lambda op: None)
            r = reference(A.buf[:, :K], B.buf[:, :K], lo(A), lo(B), alpha=0.75, bias=bias, act=act,
                          aux=aux if act >= QUICKGELU_GRAD else None, residual=res)
            bnd = bound(r, tau(K, nsplit), act, "f32", bias=bias, residual=res, alpha=0.75)
            assert ((out.double() - r["C"]).abs() <= bnd).all(), (act, nsplit)


def test_bound_catches_what_the_kernel_could_get_wrong():
    """Against the reference's own bound, a product short of its last k-block's lo.hi pass, or alpha applied after
    the bias, fails on the spiked inputs; the exact value passes."""
    M, N, K = 64, 40, 200
    a32, b32 = scaled_inputs(M, N, K, seed=1, spikes=spike_plan(M, N, K))
    (ah, al), (bh, bl) = split_hi_lo(a32), split_hi_lo(b32)
    bias = torch.randn(N, generator=torch.Generator().manual_seed(0))
    r = reference(ah, bh, al, bl, alpha=0.6875, bias=bias)
    bnd = bound(r, tau(K, 3), NONE, "f32", bias=bias, alpha=0.6875)
    assert ((r["C"].float().double() - r["C"]).abs() <= bnd).all()
    k0 = (K - 1) // 64 * 64
    short = r["C"] - 0.6875 * (al[:, k0:].double() @ bh[:, k0:].double().t())
    assert not ((short - r["C"]).abs() <= bnd).all()
    late = 0.6875 * (r["acc"] + bias.double())
    assert not ((late - r["C"]).abs() <= bnd).all()


def test_scaled_inputs_and_spikes():
    M, N, K = 300, 260, 450
    sp = spike_plan(M, N, K)
    a, b = scaled_inputs(M, N, K, seed=2, spikes=sp)
    assert a.dtype == b.dtype == torch.float32 and a.shape == (M, K) and b.shape == (N, K)
    mag = (a.abs().mean(1, keepdim=True) * b.abs().mean(1)).log2()
    assert float(mag.max() - mag.min()) > 30          # |C| spans > 2^30
    S = a.abs().double() @ b.abs().double().t()
    for i, j, k in sp:
        assert float(a[i, k].double().abs() * b[j, k].double().abs() / S[i, j]) > 0.9, (i, j, k)
    assert {i for i, _, _ in sp} >= {0, 31, 32, 127, 128, 255, 256, M - 1}
    assert {j for _, j, _ in sp} >= {0, 15, 16, 127, 128, 255, 256, N - 1}
    assert {k for _, _, k in sp} >= {0, K - 1, 448}


# ---------------------------------------------------------------------------------------- branch map
def test_branch_map_hand_cases():
    # test_gpu_ops.py's tail-split shapes: 74 CTA pairs, 256 x 256 tiles
    want = {(8224, 3072, 1024): (396, 2), (8224, 4096, 1024): (528, 4), (5082, 3072, 768): (240, 4),
            (5082, 2304, 768): (180, 2), (8224, 2000, 256): (264, 1), (8224, 2904, 512): (396, 2)}
    for (M, N, K), (tiles, f) in want.items():
        b = branches(M, N, K)
        assert (b["tiles"], b["tail_f"], b["workers"]) == (tiles, f, 74), (M, N, K, b)
        assert b["tail_first"] == tiles - (tiles % 74 if f > 1 else 0)
    b = branches(8224, 4096, 1024)
    assert b["items"] == 518 + 10 * 4 and b["rounds"] == 8 and b["acc_reuse"]
    # with max_ctas = 132 (66 pairs) the 528 tiles make 8 full rounds: nothing split
    assert branches(8224, 4096, 1024, max_ctas=132)["tail_f"] == 1
    # split-K clamp: 9 k-blocks in 4 requested slices -> 3 per slice -> 3 slices, none short
    b = branches(66, 768, 576, k_slices=4)
    assert (b["slices"], b["kb_per_slice"], b["short_last_slice"]) == (3, 3, False)
    b = branches(66, 768, 428, k_slices=3)
    assert (b["slices"], b["kb_per_slice"], b["kiters_min"], b["short_last_slice"]) == (3, 3, 1, True)
    assert branches(66, 768, 100, k_slices=8)["slices"] == 2        # no more slices than k-blocks
    assert branches(64, 64, 64, k_slices=8)["slices"] == 1
    # MN-major operands and split-K never split the tail
    assert branches(8224, 3072, 1024, a_mn=True)["tail_f"] == 1
    # BN, stages, M tails
    assert branches(100, 255, 64)["BN"] == 128 and branches(100, 256, 64)["BN"] == 256
    assert branches(100, 512, 5 * 64)["kiters_lt_stages"] and not branches(100, 512, 6 * 64)["kiters_lt_stages"]
    assert branches(100, 200, 7 * 64)["kiters_lt_stages"] and not branches(100, 200, 8 * 64)["kiters_lt_stages"]
    assert branches(100, 512, 64, nsplit=3)["kiters_lt_stages"] and not branches(100, 512, 128, nsplit=3)["kiters_lt_stages"]
    assert [branches(M, 256, 64)["m_tail"] for M in (256, 1, 128, 129, 255, 512)] == \
        ["none", "peer_empty", "peer_empty", "peer_partial", "peer_partial", "none"]
    # slabs wholly past N
    assert branches(200, 601, 130, max_ctas=4)["slab_past_n"] and not branches(200, 700, 130, max_ctas=4)["slab_past_n"]
    assert branches(200, 1029, 264, max_ctas=8)["tail_f"] == 4 and branches(200, 1029, 264, max_ctas=8)["slab_past_n"]


def _sweep_class(M, N, K, nsplit):
    b = branches(M, N, K, nsplit)
    return (b["BN"], b["m_tail"], b["m_warp_partial"], n_class(N), b["k_ragged"], b["kiters_lt_stages"])


def test_sweep_reaches_every_branch_combination():
    """The sweep's (M, N, K) list, in both modes, reaches every combination of BN, M tail (none / peer CTA empty /
    peer partial) x M % 32, N tail (full / tile / 16-column chunk / ragged float4), ragged K and k-iterations below
    the pipeline depth that any problem up to 600 x 600 x 600 reaches."""
    every = set()
    for nsplit in (1, 3):
        for M, N, K in itertools.product(range(1, 601), [64, 100, 101, 128, 130, 176, 256, 259, 276, 304, 512],
                                         [16, 64, 100, 128, 200, 448, 450, 600]):
            every.add(_sweep_class(M, N, K, nsplit))
        for N in range(1, 601):
            every.add(_sweep_class(200, N, 450, nsplit))
    got = {_sweep_class(M, N, K, ns) for M, N, K, ns in itertools.product(SWEEP_M, SWEEP_N, SWEEP_K, (1, 3))}
    assert every == got, sorted(every - got)


def test_epilogue_schedules_reach_every_scheduling_form():
    """Each scheduling form of the epilogue test is what its name says for every shape it runs, and together they
    reach: one round, several rounds with accumulator stages reused, tail split f = 2 and f = 4, a slab wholly past
    N, split-K with a short last slice, each M tail class and each N tail class."""
    seen = set()
    for name, (max_ctas, k_slices, K, ns) in SCHEDULES.items():
        for M, N in itertools.product(SCHED_M, ns):
            b = branches(M, N, K, k_slices=k_slices, max_ctas=max_ctas)
            if name == "single":
                assert b["rounds"] == 1 and b["tail_f"] == 1
            elif name == "rounds":
                assert b["rounds"] == 3 and b["acc_reuse"] and b["tail_f"] == 1
            elif name.startswith("tail"):
                assert b["tail_f"] == int(name[-1]), (name, M, N, b)
            else:
                assert b["slices"] == 3 and b["short_last_slice"] and b["k_ragged"]
            seen |= {("m", b["m_tail"]), ("n", n_class(N)), ("past", b["slab_past_n"])}
    assert seen >= {("m", "none"), ("m", "peer_empty"), ("m", "peer_partial"), ("n", "full"), ("n", "tile"),
                    ("n", "chunk16"), ("n", "ragged4"), ("past", True)}


def test_gpu_test_file_dry_runs_on_the_cpu_restatement():
    """tests/test_gpu_gemm_shapes.py itself, run by pytest on the CPU with libhba served by its restatement; left
    out: the production shapes (fp64 references of up to 50432 x 3072 x 768 are minutes of CPU time) and what the
    restatement does not restate: that the device reads the hi part's padding (the restatement reads [0, K) only)
    and bit-exact row slices or repeats (its torch matmul picks kernels by shape)."""
    tool = os.path.join(ROOT, "tests", "emulate_clip_gpu_tests.py")
    out = subprocess.run([sys.executable, tool, os.path.join(ROOT, "tests", "test_gpu_gemm_shapes.py"), "-k",
                          "not production and not zero_padded_hi and not repeated and not row_slices"],
                         capture_output=True, text=True, timeout=3000, env=dict(os.environ, OMP_NUM_THREADS="8"))
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-2000:]
    tail = [l for l in out.stdout.splitlines() if " passed" in l][-1]
    assert "failed" not in tail and "error" not in tail and int(tail.split(" passed")[0].split()[-1]) >= 400, tail
