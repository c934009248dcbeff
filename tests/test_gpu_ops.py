"""GPU parity tests of every libhba operator against the CPU oracle (oracle/ops_ref.py), through
the C-ABI (hba.ops -> ctypes -> libhba.so).  Tolerances are stated per test."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _imports():
    import hba
    from hba import ops
    from oracle import ops_ref
    return hba, ops, ops_ref


def rel_err(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def make_operand(ops, x, split, K_pad=None):
    rows, cols = x.shape
    op = ops.Operand.empty(rows, K_pad or cols, split, x.device, zero=True)
    ops.split_bf16(x.contiguous(), op)
    return op


def operand_value(op):
    """fp64 value represented by an operand (hi + lo)."""
    hi = op.buf[:, :op.K].double()
    if op.lo_off > 0:
        hi = hi + op.buf[:, op.lo_off:op.lo_off + op.K].double()
    return hi


# ----------------------------------------------------------------------------------- GEMM
@pytest.mark.parametrize("M,N,K", [(128, 256, 64), (128, 128, 64), (300, 256, 128), (256, 512, 256),
                                   (2000, 768, 512), (8224, 1024, 1024), (32, 1024, 256),
                                   (520, 1000, 192)])
@pytest.mark.parametrize("split", [False, True])
def test_gemm_plain(M, N, K, split):
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn(M, K, generator=g).to(DEV)
    b = torch.randn(N, K, generator=g).to(DEV)
    A, B = make_operand(ops, a, split), make_operand(ops, b, split)
    out = torch.full((M, _pad4(N)), float("nan"), device=DEV)[:, :N]
    ops.gemm(A, B, M, out_f32=out)
    torch.cuda.synchronize()
    if split:
        want = a.double() @ b.double().t()
        tol = 2e-5   # bf16x3: hi.hi + lo.hi + hi.lo, missing lo.lo ~ 2^-16
    else:
        want = operand_value(A) @ operand_value(B).t()  # exact product of the bf16 operands
        tol = 2e-6 * math.sqrt(K)                        # fp32 accumulation only
    assert torch.isfinite(out).all()
    assert rel_err(out, want) < tol, (rel_err(out, want), tol)


def _pad4(n):
    return (n + 3) // 4 * 4


@pytest.mark.parametrize("split", [False, True])
def test_gemm_epilogues(split):
    hba, ops, ref = _imports()
    from hba._lib import (HBA_ACT_QUICKGELU, HBA_ACT_QUICKGELU_GRAD, HBA_ACT_GELU_ERF,
                          HBA_ACT_GELU_ERF_GRAD)
    g = torch.Generator().manual_seed(5)
    M, N, K = 333, 512, 128
    a = torch.randn(M, K, generator=g).to(DEV)
    b = (torch.randn(N, K, generator=g) * 0.2).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    res = torch.randn(M, N, generator=g).to(DEV)
    aux = torch.randn(M, N, generator=g).to(DEV)
    A, B = make_operand(ops, a, split), make_operand(ops, b, split)
    base = (operand_value(A) @ operand_value(B).t()) if not split else a.double() @ b.double().t()
    tol = 3e-5 if split else 3e-5
    # bias + QuickGELU + residual, fp32 and bf16(hi/lo) outputs, pre-activation saved
    out = torch.empty(M, N, device=DEV)
    pre = torch.empty(M, N, device=DEV)
    outb = ops.Operand.empty(M, N, split, DEV)
    ops.gemm(A, B, M, bias=bias, act=HBA_ACT_QUICKGELU, residual=res, out_f32=out, out=outb,
             pre_out=pre)
    z = base + bias.double()
    want = z * torch.sigmoid(1.702 * z) + res.double()
    assert rel_err(pre, z) < tol
    assert rel_err(out, want) < tol
    assert rel_err(operand_value(outb), want) < (2e-5 if split else 5e-3)
    # bf16 pre-activation output
    preb = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    ops.gemm(A, B, M, bias=bias, out_f32=out, pre_out=preb)
    assert rel_err(preb.float(), z) < 5e-3
    # GELU(erf)
    ops.gemm(A, B, M, bias=bias, act=HBA_ACT_GELU_ERF, out_f32=out)
    assert rel_err(out, torch.nn.functional.gelu(z)) < tol
    # activation gradients: out = acc * act'(aux)
    ops.gemm(A, B, M, act=HBA_ACT_QUICKGELU_GRAD, aux=aux, out_f32=out)
    s = torch.sigmoid(1.702 * aux.double())
    assert rel_err(out, base * (s * (1 + 1.702 * aux.double() * (1 - s)))) < tol
    auxb = aux.to(torch.bfloat16)
    ops.gemm(A, B, M, act=HBA_ACT_QUICKGELU_GRAD, aux=auxb, out_f32=out)
    s = torch.sigmoid(1.702 * auxb.double())
    assert rel_err(out, base * (s * (1 + 1.702 * auxb.double() * (1 - s)))) < tol
    ops.gemm(A, B, M, act=HBA_ACT_GELU_ERF_GRAD, aux=aux, out_f32=out)
    x = aux.double()
    dg = 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
    assert rel_err(out, base * dg) < tol
    # transposed outputs (fp32 + bf16 hi/lo), alpha
    Mp = 336
    outT = torch.zeros(N, Mp, device=DEV)
    outTb = ops.Operand.empty(N, Mp, split, DEV, zero=True)
    ops.gemm(A, B, M, out_f32=outT, out=outTb, transpose_out=True, alpha=0.5)
    assert rel_err(outT[:, :M], 0.5 * base.t()) < tol
    assert rel_err(operand_value(outTb)[:, :M], 0.5 * base.t()) < (2e-5 if split else 5e-3)
    assert float(outT[:, M:].abs().max()) == 0.0


@pytest.mark.parametrize("M,N,K,slices", [(32, 1024, 4096, 8), (66, 768, 3072, 6), (66, 3072, 768, 3), (32, 768, 1024, 4)])
@pytest.mark.parametrize("split", [False, True])
def test_gemm_skinny_split_k_with_fused_epilogue(M, N, K, slices, split):
    """Row GEMMs (CLS / EOT rows) split along K: the slices write fp32 partial sums and the slice reduction runs the
    GEMM's own epilogue (bias, pre-activation output, QuickGELU / its gradient, residual, fp32 + bf16 hi/lo outputs).
    Same results as the unsplit kernel up to fp32 re-association, identical from run to run."""
    hba, ops, ref = _imports()
    from hba._lib import HBA_ACT_QUICKGELU, HBA_ACT_QUICKGELU_GRAD
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g).to(DEV)
    b = (torch.randn(N, K, generator=g) * 0.05).to(DEV)
    bias, res = torch.randn(N, generator=g).to(DEV), torch.randn(M, N, generator=g).to(DEV)
    aux = torch.randn(M, N, generator=g).to(DEV).to(torch.bfloat16)
    A, B = make_operand(ops, a, split), make_operand(ops, b, split)
    base = (operand_value(A) @ operand_value(B).t()) if not split else a.double() @ b.double().t()
    tol = 3e-5
    ws = torch.empty(slices * M * N, device=DEV)
    z = base + bias.double()
    # bias + QuickGELU + residual -> fp32 and bf16 outputs, pre-activation saved (bf16)
    out, out1 = torch.empty(M, N, device=DEV), torch.empty(M, N, device=DEV)
    pre = torch.empty(M, N, device=DEV, dtype=torch.bfloat16)
    outb = ops.Operand.empty(max(M, 128), N, split, DEV)
    ops.gemm(A, B, M, bias=bias, act=HBA_ACT_QUICKGELU, residual=res, out_f32=out, out=outb, pre_out=pre,
             k_slices=slices, k_workspace=ws)
    want = z * torch.sigmoid(1.702 * z) + res.double()
    assert rel_err(out, want) < tol
    assert rel_err(pre.float(), z) < 5e-3
    assert rel_err(operand_value(outb)[:M], want) < (2e-5 if split else 5e-3)
    ops.gemm(A, B, M, bias=bias, act=HBA_ACT_QUICKGELU, residual=res, out_f32=out1)      # unsplit kernel
    assert rel_err(out, out1) < (4e-5 if split else 1e-5)   # fp32 mode: two bf16x3 evaluations, 2e-5 each
    out2 = torch.empty(M, N, device=DEV)
    ops.gemm(A, B, M, bias=bias, act=HBA_ACT_QUICKGELU, residual=res, out_f32=out2, k_slices=slices, k_workspace=ws)
    assert torch.equal(out, out2)                                                         # fixed-order reduction
    # activation gradient with a bf16 pre-activation, bf16-only output
    gh = ops.Operand.empty(max(M, 128), N, split, DEV)
    ops.gemm(A, B, M, act=HBA_ACT_QUICKGELU_GRAD, aux=aux, out=gh, k_slices=slices, k_workspace=ws)
    s_ = torch.sigmoid(1.702 * aux.double())
    assert rel_err(operand_value(gh)[:M], base * (s_ * (1 + 1.702 * aux.double() * (1 - s_)))) < (2e-5 if split else 5e-3)
    # "auto" picks a split for these shapes
    assert ops.auto_k_slices(M, N, K, min_kblocks=4) > 1


@pytest.mark.parametrize("M,N,K,even_ctas", [(8224, 3072, 1024, 132), (8224, 4096, 1024, 132), (5082, 3072, 768, 120),
                                             (5082, 2304, 768, 120), (8224, 2000, 256, 88), (8224, 2904, 512, 132)])
def test_gemm_tail_split_is_bit_identical(M, N, K, even_ctas):
    """The partial last round of the persistent schedule is cut into 2 or 4 column slabs per tile (narrower UMMAs on
    the same accumulator columns).  Every element still sums its K products in the same order, so the result equals -
    bit for bit - a launch whose worker count divides the tile count (no partial round, nothing split), and the
    fused epilogue (bias + QuickGELU + residual, fp32 + bf16 outputs) sees the same values."""
    hba, ops, ref = _imports()
    from hba._lib import HBA_ACT_QUICKGELU
    g = torch.Generator().manual_seed(M + N)
    a = torch.randn(M, K, generator=g).to(DEV)
    b = (torch.randn(N, K, generator=g) * 0.05).to(DEV)
    bias, res = torch.randn(N, generator=g).to(DEV), torch.randn(M, N, generator=g).to(DEV)
    A, B = make_operand(ops, a, False), make_operand(ops, b, False)
    tiles = -(-M // 256) * -(-N // 256)
    assert tiles % 74 != 0 and tiles % (even_ctas // 2) == 0, "pick shapes with / without a partial round"
    outs = []
    for max_ctas in (0, even_ctas):
        o32 = torch.full((M, N), float("nan"), device=DEV)
        ob = ops.Operand.empty(M, N, False, DEV)
        ops.gemm(A, B, M, bias=bias, act=HBA_ACT_QUICKGELU, residual=res, out_f32=o32, out=ob, max_ctas=max_ctas)
        outs.append((o32, ob.buf.clone()))
    assert torch.isfinite(outs[0][0]).all()
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])
    z = operand_value(A) @ operand_value(B).t() + bias.double()
    assert rel_err(outs[0][0], z * torch.sigmoid(1.702 * z) + res.double()) < 3e-5


def test_gemm_errors():
    hba, ops, ref = _imports()
    a = ops.Operand.empty(64, 96, False, DEV)
    b = ops.Operand.empty(128, 100, False, DEV)  # row pitch not a multiple of 8 elements (16 bytes)
    with pytest.raises(RuntimeError, match="multiples of 8"):
        ops.gemm(a, b, 64, K=96, out_f32=torch.empty(64, 128, device=DEV))
    with pytest.raises(RuntimeError, match="no output"):
        ops.gemm(a, ops.Operand.empty(128, 96, False, DEV), 64)


# ----------------------------------------------------------------------------------- row-wise
@pytest.mark.parametrize("cols", [128, 256, 768, 1024])
@pytest.mark.parametrize("split", [False, True])
def test_layernorm_fwd_bwd(cols, split):
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(cols)
    rows = 77
    x = (torch.randn(rows, cols, generator=g) * 2 + 0.3).requires_grad_(True)
    w = torch.randn(cols, generator=g)
    b = torch.randn(cols, generator=g)
    y = torch.nn.functional.layer_norm(x, (cols,), w, b, 1e-5)
    dy = torch.randn(rows, cols, generator=g)
    y.backward(dy)
    xd, wd, bd = x.detach().to(DEV), w.to(DEV), b.to(DEV)
    yf = torch.empty(rows, cols, device=DEV)
    yo = ops.Operand.empty(rows, cols, split, DEV)
    ops.layernorm_fwd(xd, rows, cols, wd, bd, 1e-5, y_f32=yf, y=yo)
    assert rel_err(yf, y.detach()) < 1e-5
    assert rel_err(operand_value(yo), y.detach()) < (2e-5 if split else 5e-3)
    dx = torch.empty(rows, cols, device=DEV)
    ops.layernorm_bwd(dy.to(DEV), xd, rows, cols, wd, 1e-5, dx)
    assert rel_err(dx, x.grad) < 2e-5
    prev = torch.randn(rows, cols, generator=g).to(DEV)
    dx2 = prev.clone()
    ops.layernorm_bwd(dy.to(DEV), xd, rows, cols, wd, 1e-5, dx2, accumulate=True)
    assert rel_err(dx2, x.grad + prev.cpu()) < 2e-5
    # strided row selection (CLS rows): every 5th row
    ysel = torch.empty(rows // 5, cols, device=DEV)
    ops.layernorm_fwd(xd, rows // 5, cols, wd, bd, 1e-5, row_step=5, y_f32=ysel)
    assert rel_err(ysel, y.detach()[::5][: rows // 5]) < 1e-5


@pytest.mark.parametrize("split", [False, True])
def test_patch_embed_front_end(split):
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(3)
    B, P, width, res = 3, 14, 256, 224
    img = torch.randn(B, 3, res, res, generator=g)
    conv = torch.nn.Conv2d(3, width, P, P, bias=False)
    cls = torch.randn(width, generator=g)
    pos = torch.randn(257, width, generator=g)
    gam, bet = torch.randn(width, generator=g), torch.randn(width, generator=g)
    with torch.no_grad():
        c = conv(img).reshape(B, width, -1).permute(0, 2, 1)
        xr = torch.cat([cls.expand(B, 1, width), c], 1) + pos
        xr = torch.nn.functional.layer_norm(xr, (width,), gam, bet, 1e-5).reshape(B * 257, width)
    kp = 640
    patches = ops.Operand.empty(B * 256, kp, split, DEV, zero=True)
    ops.im2col_patches(img.to(DEV), P, patches)
    wop = make_operand(ops, conv.weight.detach().reshape(width, -1).to(DEV), split, K_pad=kp)
    co = torch.empty(B * 256, width, device=DEV)
    ops.gemm(patches, wop, B * 256, out_f32=co)
    x = torch.empty(B * 257, width, device=DEV)
    ops.assemble_tokens_ln(co, B, 256, width, cls.to(DEV), pos.to(DEV), gam.to(DEV), bet.to(DEV),
                           1e-5, x)
    assert rel_err(x, xr) < (1e-4 if split else 2e-2)


def test_embed_and_gather():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(4)
    S, T, w = 5, 77, 128
    tok = torch.randint(0, 1000, (S, T), generator=g)
    table, pos = torch.randn(1000, w, generator=g), torch.randn(T, w, generator=g)
    x = torch.empty(S * T, w, device=DEV)
    ops.embed_tokens(tok.to(DEV), table.to(DEV), pos.to(DEV), x)
    assert torch.equal(x.cpu(), (table[tok] + pos).reshape(S * T, w))
    idx = torch.tensor([3, 0, 100, 384])
    out = torch.empty(4, w, device=DEV)
    ops.gather_rows(x, idx.to(DEV), w, out)
    assert torch.equal(out.cpu(), x.cpu()[idx])


# ----------------------------------------------------------------------------------- attention
@pytest.mark.parametrize("B,T,H,causal", [(2, 257, 4, False), (3, 77, 2, True), (2, 197, 3, False),
                                          (1, 50, 1, False)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_attention_fwd(B, T, H, causal, dtype):
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(T)
    d = H * 64
    qkv = torch.randn(B * T, 3 * d, generator=g).to(dtype)
    want = ref.attention(qkv.float(), B, T, H, causal)
    out = ops.Operand.empty(B * T, d, True, DEV)
    of = torch.empty(B * T, d, device=DEV)
    ops.attention_fwd(qkv.to(DEV), B, T, H, causal=causal, out=out, out_f32=of)
    assert rel_err(of, want) < 2e-5
    assert rel_err(operand_value(out), want) < 2e-5
    if dtype == torch.bfloat16:
        # tensor-core path (tcgen05, P rounded to bf16): hi-only output, stated tolerance 1e-2
        outb = ops.Operand.empty(B * T, d, False, DEV)
        of2 = torch.full((B * T, d), float("nan"), device=DEV)
        ops.attention_fwd(qkv.to(DEV), B, T, H, causal=causal, out=outb, out_f32=of2)
        assert torch.isfinite(of2).all()
        assert rel_err(of2, want) < 1e-2, rel_err(of2, want)
        assert rel_err(operand_value(outb), want) < 1.5e-2
    if not causal:
        o0 = torch.empty(B, d, device=DEV)
        ops.attention_fwd(qkv.to(DEV), B, T, H, first_row_only=True, out_f32=o0)
        assert rel_err(o0, want.view(B, T, d)[:, 0]) < 2e-5


def test_attention_bwd_row0():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(11)
    B, T, H = 3, 257, 2
    d = H * 64
    qkv = torch.randn(B * T, 3 * d, generator=g, dtype=torch.float64).requires_grad_(True)
    o = ref.attention(qkv, B, T, H).view(B, T, d)[:, 0]
    do = torch.randn(B, d, generator=g, dtype=torch.float64)
    o.backward(do)
    dq = torch.full((B * T, 3 * d), float("nan"), device=DEV)
    ops.attention_bwd_row0(qkv.detach().float().to(DEV), B, T, H, do.float().to(DEV), dq)
    assert rel_err(dq, qkv.grad) < 2e-5


# ----------------------------------------------------------------------------------- DoRA
@pytest.mark.parametrize("in_f,out_f,r", [(1024, 1024, 32), (768, 768, 32), (256, 256, 8)])
@pytest.mark.parametrize("split", [False, True])
def test_dora_merge_fwd_bwd(in_f, out_f, r, split):
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(in_f + r)
    W0 = torch.randn(out_f, in_f, generator=g) * 0.03
    m0, D = ref.dora_init(W0)
    bound_a, bound_b = 1 / math.sqrt(out_f), 1 / math.sqrt(r)
    A = ((torch.rand(r, out_f, generator=g) * 2 - 1) * bound_a).double().requires_grad_(True)
    Bm = ((torch.rand(in_f, r, generator=g) * 2 - 1) * bound_b).double().requires_grad_(True)
    m = (m0 * (1 + 0.1 * torch.randn(out_f, generator=g))).double().requires_grad_(True)
    scale = 16 / r
    W = ref.dora_weight(D.double(), A, Bm, m, scale)
    G = torch.randn(out_f, in_f, generator=g, dtype=torch.float64)
    (W * G).sum().backward()
    Dd = D.contiguous().to(DEV)
    Ad, Bd, md = A.detach().float().to(DEV), Bm.detach().float().to(DEV), m.detach().float().to(DEV)
    w_t = torch.empty(in_f, out_f, device=DEV)
    w = ops.Operand.empty(out_f, in_f, split, DEV)
    wt = ops.Operand.empty(in_f, out_f, split, DEV)
    nrm = torch.empty(out_f, device=DEV)
    ops.dora_merge_fwd(Dd, Ad, Bd, md, scale, 1e-8, w_t_f32=w_t, w=w, wt=wt, norm_out=nrm)
    assert rel_err(w_t.t(), W.detach()) < 2e-6
    assert rel_err(operand_value(w), W.detach()) < (2e-5 if split else 5e-3)
    assert rel_err(operand_value(wt), W.detach().t()) < (2e-5 if split else 5e-3)
    dm, dA, dB = torch.empty_like(md), torch.empty_like(Ad), torch.empty_like(Bd)
    ws = torch.empty(in_f, out_f, device=DEV)
    ops.dora_merge_bwd(G.float().to(DEV), Dd, Ad, Bd, md, scale, 1e-8, dm, dA, dB, ws)
    assert rel_err(dm, m.grad) < 2e-5
    assert rel_err(dA, A.grad) < 2e-5
    assert rel_err(dB, Bm.grad) < 2e-5


def test_dora_layer_module_matches_oracle():
    """hba.DoRALayer (fused kernels + autograd.Function) == reference formula under autograd."""
    hba, ops, ref = _imports()
    torch.manual_seed(0)
    lin = torch.nn.Linear(256, 256)
    torch.manual_seed(1)
    layer = hba.DoRALayer(lin, r=32).to(DEV)
    W = layer.weight
    G = torch.randn(256, 256, device=DEV)
    (W * G).sum().backward()
    A = layer.delta_D_A.detach().cpu().double().requires_grad_(True)
    Bm = layer.delta_D_B.detach().cpu().double().requires_grad_(True)
    m = layer.m.detach().cpu().double().requires_grad_(True)
    Wr = ref.dora_weight(layer.D.cpu().double(), A, Bm, m, layer.scaling)
    (Wr * G.cpu().double()).sum().backward()
    assert rel_err(W.detach(), Wr.detach()) < 2e-6
    assert rel_err(layer.m.grad, m.grad) < 2e-5
    assert rel_err(layer.delta_D_A.grad, A.grad) < 2e-5
    assert rel_err(layer.delta_D_B.grad, Bm.grad) < 2e-5


# ----------------------------------------------------------------------------------- heads
def test_cos_head_fwd_bwd():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(2)
    B, Cc, E = 32, 66, 768
    img = torch.randn(B, E, generator=g, dtype=torch.float64).requires_grad_(True)
    txt = torch.randn(Cc, E, generator=g, dtype=torch.float64).requires_grad_(True)
    ls = torch.tensor(math.log(100.0), dtype=torch.float64)
    tgt = torch.randn(B, Cc, generator=g, dtype=torch.float64) * 9.5 + 5.75
    pred = ref.cos_logits(img, txt, ls)
    loss = torch.nn.functional.mse_loss(pred, tgt)
    loss.backward()
    imgd, txtd = img.detach().float().to(DEV), txt.detach().float().to(DEV)
    lsd, tgtd = ls.float().reshape(1).to(DEV), tgt.float().to(DEV)
    p = torch.empty(B, Cc, device=DEV)
    l = torch.empty(1, device=DEV)
    ops.cos_head_fwd(imgd, txtd, lsd, p, tgtd, l)
    assert rel_err(p, pred.detach()) < 1e-5
    assert abs(float(l) - float(loss)) / float(loss) < 1e-5
    di, dt = torch.empty(B, E, device=DEV), torch.empty(Cc, E, device=DEV)
    ops.cos_head_bwd(imgd, txtd, lsd, di, dt, pred=p, target=tgtd)  # fused MSE gradient
    assert rel_err(di, img.grad) < 2e-4
    assert rel_err(dt, txt.grad) < 2e-4
    dp = (2 * (pred.detach() - tgt) / (B * Cc)).float().to(DEV)
    ops.cos_head_bwd(imgd, txtd, lsd, di, dt, d_pred=dp)
    assert rel_err(di, img.grad) < 2e-4
    assert rel_err(dt, txt.grad) < 2e-4


@pytest.mark.parametrize("B,Cc,E,G,shared", [(32, 66, 768, 1, False), (4, 66, 768, 3, False), (32, 66, 768, 4, True),
                                             (7, 5, 128, 2, False), (20, 9, 1024, 2, False)])
def test_cos_mse_fused_single_launch(B, Cc, E, G, shared):
    """hba_cos_mse_fwd / _bwd: logits + nn.MSELoss + non-finite flag + running sums in one launch per direction,
    for G independent groups (lock-stepped conditions) with per-group or shared targets; upstream d_loss."""
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(B + Cc + G)
    img = torch.randn(G, B, E, generator=g, dtype=torch.float64).requires_grad_(True)
    txt = torch.randn(G, Cc, E, generator=g, dtype=torch.float64).requires_grad_(True)
    ls = torch.tensor(math.log(100.0), dtype=torch.float64)
    tgt = torch.randn(1 if shared else G, B, Cc, generator=g, dtype=torch.float64) * 9.5 + 5.75
    up = torch.rand(G, generator=g, dtype=torch.float64) + 0.5
    losses = []
    for k in range(G):
        pred = ref.cos_logits(img[k], txt[k], ls)
        losses.append(torch.nn.functional.mse_loss(pred, tgt[0 if shared else k]))
    (torch.stack(losses) * up).sum().backward()
    f = lambda t: t.detach().float().to(DEV).contiguous()
    imgd, txtd, tgtd = f(img).view(G * B, E), f(txt).view(G * Cc, E), f(tgt)
    lsd = ls.float().reshape(1).to(DEV)
    p = torch.empty(G * B, Cc, device=DEV)
    loss = torch.empty(G, device=DEV)
    bad_step = torch.full((G,), 7, dtype=torch.int32, device=DEV)
    bad_total = torch.zeros(G, dtype=torch.int32, device=DEV)
    total = torch.zeros(G, dtype=torch.float64, device=DEV)
    ws = torch.zeros(G * (B + 1), device=DEV)
    stride = 0 if shared else B * Cc
    for rep in range(3):   # the workspace is left ready for the next launch
        ops.cos_mse_fwd(imgd, txtd, lsd, p, B=B, groups=G, target=tgtd, target_group_stride=stride, loss=loss,
                        bad_step=bad_step, bad_total=bad_total, total=total, workspace=ws)
    torch.cuda.synchronize()
    want = torch.stack(losses).detach()
    assert rel_err(loss, want) < 1e-5
    assert bad_step.tolist() == [0] * G and bad_total.tolist() == [0] * G
    assert rel_err(total, 3 * B * want) < 1e-5
    first = loss.clone()
    ops.cos_mse_fwd(imgd, txtd, lsd, p, B=B, groups=G, target=tgtd, target_group_stride=stride, loss=loss,
                    bad_step=bad_step, bad_total=bad_total, total=total, workspace=ws)
    assert torch.equal(loss, first)                       # fixed-order reduction: run-to-run identical
    di, dt = torch.empty(G * B, E, device=DEV), torch.empty(G * Cc, E, device=DEV)
    ops.cos_mse_bwd(imgd, txtd, lsd, p, tgtd, di, dt, B=B, groups=G, target_group_stride=stride, d_loss=f(up))
    assert rel_err(di.view(G, B, E), img.grad) < 2e-4
    assert rel_err(dt.view(G, Cc, E), txt.grad) < 2e-4
    # a non-finite target in the last group: flagged, counted, not accumulated; the other groups unaffected
    if not shared:
        before = total.clone()
        tgtd[G - 1, 0, 0] = float("nan")
        ops.cos_mse_fwd(imgd, txtd, lsd, p, B=B, groups=G, target=tgtd, target_group_stride=stride, loss=loss,
                        bad_step=bad_step, bad_total=bad_total, total=total, workspace=ws)
        assert bad_step.tolist() == [0] * (G - 1) + [1] and bad_total.tolist() == [0] * (G - 1) + [1]
        assert float(total[G - 1]) == float(before[G - 1])
        if G > 1:
            assert rel_err(total[:G - 1] - before[:G - 1], B * want[:G - 1]) < 1e-5
        # evaluate_model's form (no flag): accumulated unconditionally
        ops.cos_mse_fwd(imgd, txtd, lsd, p, B=B, groups=G, target=tgtd, target_group_stride=stride, loss=loss,
                        total=total, workspace=ws)
        assert math.isnan(float(total[G - 1]))


def test_softmax_ce():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(8)
    B, Cc = 37, 1000
    z = (torch.randn(B, Cc, generator=g) * 3).requires_grad_(True)
    y = torch.randint(0, Cc, (B,), generator=g)
    loss = torch.nn.functional.cross_entropy(z, y)
    loss.backward()
    l = torch.empty(1, device=DEV)
    dz = torch.empty(B, Cc, device=DEV)
    hit = torch.empty(1, device=DEV, dtype=torch.int32)
    ws = torch.empty(2 * B, device=DEV)
    ops.softmax_ce(z.detach().to(DEV), y.to(DEV), l, dz, hit, ws)
    assert abs(float(l) - float(loss)) < 1e-5 * abs(float(loss))
    assert rel_err(dz, z.grad) < 1e-5
    assert int(hit) == int((z.argmax(1) == y).sum())


# ----------------------------------------------------------------------------------- optimisers
def _ptr_table(tensor_lists):
    n = len(tensor_lists[0])
    flat = []
    for i in range(n):
        for lst in tensor_lists:
            flat.append(lst[i].data_ptr())
    sizes = [t.numel() for t in tensor_lists[0]]
    return (torch.tensor(flat, dtype=torch.int64, device=DEV),
            torch.tensor(sizes, dtype=torch.int64, device=DEV), n, sum(sizes))


def test_adamw_multi_matches_torch():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(9)
    shapes = [(1024,), (32, 1024), (1024, 32), (768,), (5, 7)]
    params = [torch.randn(*s, generator=g) for s in shapes]
    steps = [[torch.randn(*s, generator=g) for s in shapes] for _ in range(5)]
    want, _ = ref.adamw_reference(params, steps, lr=3e-4)
    p = [t.clone().to(DEV) for t in params]
    gr = [torch.empty_like(t) for t in p]
    m = [torch.zeros_like(t) for t in p]
    v = [torch.zeros_like(t) for t in p]
    table, sizes, n, total = _ptr_table([p, gr, m, v])
    flag = torch.zeros(1, dtype=torch.int32, device=DEV)
    for k, grads in enumerate(steps):
        for dst, src in zip(gr, grads):
            dst.copy_(src)
        ops.adamw_multi(table, sizes, n, total, 3e-4, 0.9, 0.999, 1e-8, 0.01, k + 1, flag)
    for a, b in zip(p, want):
        assert rel_err(a, b) < 1e-6
    flag.fill_(1)  # skip flag: nothing changes
    before = [t.clone() for t in p]
    ops.adamw_multi(table, sizes, n, total, 3e-4, 0.9, 0.999, 1e-8, 0.01, 6, flag)
    for a, b in zip(p, before):
        assert torch.equal(a, b)


def test_sgd_multi_matches_torch():
    hba, ops, ref = _imports()
    g = torch.Generator().manual_seed(10)
    shapes = [(300,), (17, 33)]
    params = [torch.nn.Parameter(torch.randn(*s, generator=g)) for s in shapes]
    opt = torch.optim.SGD(params, lr=0.1, momentum=0.9, weight_decay=1e-4)
    p = [t.detach().clone().to(DEV) for t in params]
    gr = [torch.empty_like(t) for t in p]
    buf = [torch.zeros_like(t) for t in p]
    table, sizes, n, total = _ptr_table([p, gr, buf])
    for k in range(4):
        grads = [torch.randn(*s, generator=g) for s in shapes]
        for q, gg, dst in zip(params, grads, gr):
            q.grad = gg.clone()
            dst.copy_(gg)
        opt.step()
        ops.sgd_multi(table, sizes, n, total, 0.1, 0.9, 1e-4, k == 0)
    for a, b in zip(p, params):
        assert rel_err(a, b.detach()) < 1e-6


# ----------------------------------------------------------------------------------- RSA
@pytest.mark.parametrize("N,Dm", [(48, 66), (200, 66), (48, 768)])
def test_rdm_matches_numpy(N, Dm):
    hba, ops, ref = _imports()
    rng = np.random.default_rng(N + Dm)
    E = rng.standard_normal((N, Dm)).astype(np.float32)
    want = 1 - np.corrcoef(E)
    np.fill_diagonal(want, 0)
    rdm = torch.empty(N, N, dtype=torch.float64, device=DEV)
    tri = torch.empty(N * (N - 1) // 2, dtype=torch.float64, device=DEV)
    ops.rdm_f64(torch.from_numpy(E).to(DEV), rdm, tri)
    assert np.abs(rdm.cpu().numpy() - want).max() < 1e-12
    assert np.abs(tri.cpu().numpy() - want[np.triu_indices(N, k=1)]).max() < 1e-12


@pytest.mark.parametrize("n", [1, 7, 1128, 2048, 2049, 5000, 100_000, 1_717_731])
def test_rank_avg_bit_exact(n):
    hba, ops, ref = _imports()
    rng = np.random.default_rng(n)
    x = rng.standard_normal(n)
    if n > 4:  # ties (incl. -0.0 == +0.0, long runs) and extreme values
        x[rng.integers(0, n, n // 3)] = np.round(x[rng.integers(0, n, n // 3)], 1)
        x[: n // 10] = 0.25
        x[-2:] = [0.0, -0.0]
        x[n // 2] = 1e300
        x[n // 2 + 1] = -1e300
    want = ref.rankdata_average(x)
    r = torch.empty(n, dtype=torch.float64, device=DEV)
    ops.rank_avg_f64(torch.from_numpy(x).to(DEV), r)
    assert np.array_equal(r.cpu().numpy(), want)


@pytest.mark.parametrize("N", [48, 300])
def test_spearman_pipeline(N):
    hba, ops, ref = _imports()
    from hba import rsa
    rng = np.random.default_rng(N)
    E = rng.standard_normal((N, 66)).astype(np.float32)
    ref_rdm = 1 - np.corrcoef(rng.standard_normal((N, 66)) + 0.5 * E)
    np.fill_diagonal(ref_rdm, 0)
    rho_w, p_w, rdm_w = ref.rdm_and_spearman(E, ref_rdm)
    rho, p, rdm = rsa.rsa_from_embeddings(torch.from_numpy(E).to(DEV), ref_rdm)
    assert abs(rho - rho_w) < 1e-10       # north star: within 1e-4
    assert abs(p - p_w) <= 1e-9 * max(p_w, 1e-300) + 1e-300
    assert np.abs(rdm - rdm_w).max() < 1e-12


@pytest.mark.parametrize("N", [48, 300])
@pytest.mark.parametrize("bad", ["nan_row", "constant_row"])
def test_rsa_nan_semantics(N, bad):
    """A diverged model (NaN or constant embedding row) must log nan, as numpy.corrcoef / scipy.stats.spearmanr do
    (NEW:625-652) - never rho = -1 (CUDA fmin/fmax drop NaN).  N=48 takes the three-kernel path, N=300 the fused
    RSA-at-scale chain."""
    from scipy.stats import spearmanr
    from hba import rsa
    rng = np.random.default_rng(N)
    E = rng.standard_normal((N, 66)).astype(np.float32)
    if bad == "nan_row":
        E[3, 5] = np.nan
    else:
        E[7] = 0.25
    ref_rdm = 1 - np.corrcoef(rng.standard_normal((N, 66)))
    np.fill_diagonal(ref_rdm, 0)
    with np.errstate(all="ignore"):
        want_rdm = 1 - np.corrcoef(E)
        np.fill_diagonal(want_rdm, 0)
        want_rho = spearmanr(ref_rdm[np.triu_indices(N, 1)], want_rdm[np.triu_indices(N, 1)])[0]
    assert math.isnan(want_rho)
    rho, p, rdm = rsa.rsa_from_embeddings(torch.from_numpy(E).to(DEV), ref_rdm)
    assert math.isnan(rho) and math.isnan(p)
    assert np.array_equal(np.isnan(rdm), np.isnan(want_rdm))
