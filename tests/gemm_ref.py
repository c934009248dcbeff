"""fp64 reference of hba_gemm_bf16, the branch map of its launcher, and inputs that expose a wrong tile.

`reference()` computes C = epilogue(A . B^T) in fp64 from the exact values handed to the kernel (the bf16 hi and lo
parts of both operands, K-major or MN-major), applying the epilogue in the order include/hba.h documents: alpha,
bias, pre_out, act or act'(aux), residual.  In fp32 mode (nsplit == 3) the product is hi.hi + lo.hi + hi.lo, the
lo.lo term dropped as in the kernel.  With it come the per-element scale S = |A| . |B|^T and the pieces a
per-element error bound needs (`bound()`; its derivation is in tests/test_gpu_gemm_shapes.py).

`branches()` restates, line by line, how the launcher (vit-project_b200/csrc/gemm_tc.cu) turns (M, N, K, ...) into
tiles, workers, rounds, tail slabs, k-blocks and split-K slices.  `scaled_inputs()` builds operands whose rows of A
and columns of B are scaled over about 2^-10 .. 2^10, with optional dominant products at chosen (row, column, k).
"""
from __future__ import annotations

import math

import torch

BM, BK = 128, 64
NUM_SMS = 148                      # B200
U32 = 2.0 ** -24                   # unit roundoff of fp32 (round to nearest)
ULP32 = 2.0 ** -23                 # one fp32 ulp relative: the most a truncating addition loses
NONE, QUICKGELU, GELU, QUICKGELU_GRAD, GELU_GRAD = range(5)
GRAD_ACTS = (QUICKGELU_GRAD, GELU_GRAD)
SQRT2 = math.sqrt(2.0)


# ---------------------------------------------------------------------------------------- activations (fp64)
def _phi(x):
    return torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)


def _cdf(x):
    return 0.5 * (1 + torch.erf(x / SQRT2))


def quickgelu_grad(a):
    s = torch.sigmoid(1.702 * a)
    return s * (1 + 1.702 * a * (1 - s))


def gelu_grad(a):
    return _cdf(a) + a * _phi(a)


def apply_act(act, z, aux=None):
    if act == NONE:
        return z
    if act == QUICKGELU:
        return z * torch.sigmoid(1.702 * z)
    if act == GELU:
        return z * _cdf(z)
    if act == QUICKGELU_GRAD:
        return z * quickgelu_grad(aux)
    if act == GELU_GRAD:
        return z * gelu_grad(aux)
    raise ValueError(act)


def act_slope(act, z, aux=None):
    """|d C / d z|: how much an error in the pre-activation z moves the output."""
    if act == NONE:
        return torch.ones_like(z)
    if act == QUICKGELU:
        return quickgelu_grad(z).abs()
    if act == GELU:
        return gelu_grad(z).abs()
    return (quickgelu_grad(aux) if act == QUICKGELU_GRAD else gelu_grad(aux)).abs()


def sfu_error(act, z, aux=None):
    """Bound on the error of the kernel's fp32 / SFU evaluation of the activation at an exact argument
    (gemm_tc.cu:78-115), absolute, per element.
      QuickGELU  v / (1 + ex2(-1.702 log2e v)): ex2.approx 2 ulp, __fdividef 2 ulp, and the rounded argument
                 moves exp by u |1.702 v| relative -> |v| (2^-20 + 1.702 |v| u).
      GELU       relu(v) - |v| h(|v|), h = 0.5 erfc: Abramowitz-Stegun 7.1.26 is good to 1.5e-7 in erf, 7.5e-8 in h;
                 the rcp / ex2 approximations and five FMAs cost <= 12 ulp of h, the rounded v^2 / 2 another
                 u v^2 of h -> |v| (7.5e-8 + h (12 ulp + u v^2)) + u |gelu(v)|.
      *_GRAD     v times the same analysis of the derivative at a = aux (exact: aux is stored in the type
                 the kernel reads)."""
    av = z.abs()
    if act == NONE:
        return torch.zeros_like(z)
    if act == QUICKGELU:
        return av * (2.0 ** -20 + 1.702 * av * U32)
    if act == GELU:
        h = 0.5 * torch.erfc(av / SQRT2)
        return av * (7.5e-8 + h * (12 * ULP32 + U32 * z * z)) + U32 * apply_act(GELU, z).abs()
    a = aux
    aa = a.abs()
    if act == QUICKGELU_GRAD:
        s = torch.sigmoid(1.702 * a)
        ds = 2.0 ** -21 + 1.702 * aa * U32
        return av * (s * (1 + 1.702 * aa)) * (ds + 4 * U32)
    h = 0.5 * torch.erfc(aa / SQRT2)
    d = (7.5e-8 + h * (12 * ULP32 + U32 * a * a) + (a * _phi(a)).abs() * (2.0 ** -21 + U32 * a * a)
         + 2 * U32 * (gelu_grad(a).abs() + 1))
    return av * d


# ---------------------------------------------------------------------------------------- reference
def _logical(x, mn, K):
    """operand -> [rows, K] fp64 (an MN-major operand is stored [K, rows])."""
    if x is None:
        return None
    x = x.double()
    return x[:K].t() if mn else x[:, :K]


def reference(a_hi, b_hi, a_lo=None, b_lo=None, *, a_mn=False, b_mn=False, K=None, alpha=1.0, bias=None,
              act=NONE, aux=None, residual=None):
    """fp64 epilogue(A . B^T) of the exact operand values.  a_hi / a_lo are [M, >= K] (K-major) or [>= K, M]
    (MN-major), likewise b_* with N; the lo parts only in fp32 mode.  Returns a dict:
      acc   the product (hi.hi + lo.hi + hi.lo in fp32 mode)
      z     alpha * acc + bias: the pre-activation (what pre_out receives)
      C     act(z) or z * act'(aux), plus residual
      S     |alpha| (|a_hi| + |a_lo|) . (|b_hi| + |b_lo|)^T: the sum of the magnitudes the kernel adds up
      aux   aux in fp64 (None without one)
      full  fp32 mode: the product of the unsplit values (hi + lo)(hi + lo)^T
      lolo  fp32 mode: |a_lo| . |b_lo|^T, which bounds |acc - full|"""
    if K is None:
        K = a_hi.shape[0] if a_mn else a_hi.shape[1]
    ah, bh = _logical(a_hi, a_mn, K), _logical(b_hi, b_mn, K)
    al, bl = _logical(a_lo, a_mn, K), _logical(b_lo, b_mn, K)
    res = {}
    acc = ah @ bh.t()
    if al is not None:
        acc = acc + al @ bh.t() + ah @ bl.t()
        res["full"] = (ah + al) @ (bh + bl).t()
        res["lolo"] = al.abs() @ bl.abs().t()
        s = (ah.abs() + al.abs()) @ (bh.abs() + bl.abs()).t()
    else:
        s = ah.abs() @ bh.abs().t()
    z = alpha * acc
    if bias is not None:
        z = z + bias.double()
    a64 = aux.double() if aux is not None else None
    c = apply_act(act, z, a64)
    if residual is not None:
        c = c + residual.double()
    res.update(acc=acc, z=z, C=c, S=abs(alpha) * s, aux=a64)
    return res


def tau(K, nsplit, slices=1):
    """Relative accumulation bound: |acc_kernel - acc| <= tau * S.  The kernel adds nsplit * K exact products
    (a bf16 x bf16 product fits fp32) into an fp32 accumulator, and the split-K reduction adds `slices` partial
    sums; each addition loses at most one fp32 ulp of the running magnitude (2^-23 even if the tensor pipe
    truncates instead of rounding), which the partial sums of |products| bound by S."""
    return ULP32 * (nsplit * K + slices)


OUT_ROUNDING = {"f32": 0.0, "bf16": 2.0 ** -8, "hilo": 2.0 ** -16}   # bf16 keeps 8 significant bits


def bound(ref, tau_, act=NONE, out="f32", bias=None, residual=None, alpha=1.0, pre=False):
    """Per-element bound on |kernel - ref["C"]| (or on |pre_out - ref["z"]| with pre=True) for an output stored
    as `out` ("f32", "bf16" hi only, "hilo" hi + lo)."""
    z = ref["z"]
    # pre-activation: accumulation, then one rounding each for alpha * acc and + bias
    ez = tau_ * ref["S"] + 2 * U32 * ((alpha * ref["acc"]).abs() + (bias.double().abs() if bias is not None else 0))
    if pre:
        return ez + OUT_ROUNDING[out] * z.abs()
    c = ref["C"]
    e = act_slope(act, z, ref["aux"]) * ez + sfu_error(act, z, ref["aux"]) + ez * ez
    e = e + 2 * U32 * c.abs()                                   # the activation's own product, the residual add
    if residual is not None:
        e = e + U32 * residual.double().abs()
    return e + OUT_ROUNDING[out] * (c.abs() + e)


# ---------------------------------------------------------------------------------------- branch map
def k_stages(BN):
    """GemmCfg<BN>::kStages (gemm_tc.cu:42): smem ring stages of 16 KB of A plus (BN / 2) x 64 of B."""
    return min(8, (192 * 1024) // (BM * BK * 2 + (BN // 2) * BK * 2))


def branches(M, N, K, nsplit=1, a_mn=False, b_mn=False, k_slices=1, max_ctas=0, num_sms=NUM_SMS):
    """What hba_gemm_bf16 / launch_gemm do with a problem (gemm_tc.cu line numbers)."""
    BN = 256 if N >= 256 else 128                                   # :903 `wide`
    TM = 2 * BM                                                      # a CTA pair's tile rows
    kblocks = -(-K // BK)                                            # :875
    slices = min(max(k_slices, 1), kblocks)                          # :876-877
    kb_per = kblocks
    if slices > 1:                                                   # :884-886 every slice owns >= 1 k-block
        kb_per = -(-kblocks // slices)
        slices = -(-kblocks // kb_per)
    last_slice_kb = kblocks - (slices - 1) * kb_per
    m_tiles, n_tiles = -(-M // TM), -(-N // BN)
    tiles = m_tiles * n_tiles                                        # :770
    workers = num_sms // 2                                           # :771-773
    if max_ctas > 0 and max_ctas // 2 < workers:
        workers = max(max_ctas // 2, 1)
    if tiles * slices < workers:
        workers = tiles * slices
    f, tail_first = 1, tiles                                         # :778-794 tail split
    if BN == 256 and slices == 1 and not a_mn and not b_mn and tiles > workers and tiles % workers:
        rem = tiles % workers
        cost2 = -(-(rem * 2) // workers) * 0.75
        cost4 = -(-(rem * 4) // workers) * 0.65
        if cost2 < 1.0 - 0.05 and cost2 <= cost4:
            f = 2
        elif cost4 < 1.0 - 0.05:
            f = 4
        if f > 1:
            tail_first = tiles - rem
    items = tail_first + (tiles - tail_first) * f if f > 1 else tiles * slices   # :475-476
    per_worker = -(-items // workers)
    slab_past_n = any((t % n_tiles) * BN + s * (BN // f) >= N for t in range(tail_first, tiles) for s in range(f))
    m_rem = M % TM
    return {
        "BN": BN, "m_tiles": m_tiles, "n_tiles": n_tiles, "tiles": tiles, "workers": workers, "items": items,
        "rounds": per_worker, "acc_reuse": per_worker > 2,
        "tail_f": f, "tail_first": tail_first, "slab_past_n": slab_past_n,
        "kblocks": kblocks, "k_ragged": K % BK != 0,
        "kiters_min": last_slice_kb * nsplit, "kiters_lt_stages": last_slice_kb * nsplit < k_stages(BN),
        "slices": slices, "kb_per_slice": kb_per, "short_last_slice": slices > 1 and last_slice_kb < kb_per,
        "m_tail": "none" if m_rem == 0 else ("peer_empty" if m_rem <= BM else "peer_partial"),
        "m_warp_partial": M % 32 != 0,
        "n_mod_bn": N % BN, "n_mod16": N % 16, "n_mod4": N % 4,
    }


def n_class(N):
    """The N-tail class: a full last tile, a partial tile of whole 16-column chunks, a partial chunk of whole
    float4 granules, or ragged columns (the element-wise path of epilogue_chunk_coalesced)."""
    BN = 256 if N >= 256 else 128
    if N % 4:
        return "ragged4"
    if N % 16:
        return "chunk16"
    return "tile" if N % BN else "full"


# ---------------------------------------------------------------------------------------- inputs
def scaled_inputs(M, N, K, *, seed=0, spikes=(), span=10):
    """fp32 A [M, K] and B [N, K]: N(0, 1) entries, row i of A scaled by 2^r_i / sqrt(K) and row j of B by 2^c_j
    with r, c uniform integers in [-span, span], so |C[i, j]| ~ 2^(r_i + c_j) varies over 2^(4 span) and an error
    normalised by max |C| cannot hide a wrong tile.  Each (i, j, k) in `spikes` makes A[i, k] B[j, k] dominant in C[i, j]:
    A[i, k] = +-8 sqrt(K) 2^r_i and B[j, k] = +-8 sqrt(K) 2^c_j, 64 K times the typical product, which is more
    than 90 % of S[i, j].  Each row and each column may appear in one spike only."""
    g = torch.Generator().manual_seed(seed)
    rows = [s[0] for s in spikes]
    cols = [s[1] for s in spikes]
    assert len(set(rows)) == len(rows) and len(set(cols)) == len(cols), spikes
    r = torch.randint(-span, span + 1, (M, 1), generator=g).double()
    c = torch.randint(-span, span + 1, (N, 1), generator=g).double()
    a = torch.randn(M, K, generator=g, dtype=torch.float64)
    b = torch.randn(N, K, generator=g, dtype=torch.float64)
    big = 8 * math.sqrt(K)
    for i, j, k in spikes:
        assert 0 <= i < M and 0 <= j < N and 0 <= k < K, (M, N, K, i, j, k)
        a[i, k] = big * (1 if (i + k) % 2 else -1)
        b[j, k] = big * (1 if (j + k) % 3 else -1)
    return (a * torch.exp2(r) / math.sqrt(K)).float(), (b * torch.exp2(c)).float()


def spike_plan(M, N, K, ks=None):
    """(row, column, k) triples for a problem: rows at the edges of the 32-row epilogue warps, the 128-row CTA
    halves and the 256-row tiles plus the last row; columns at the edges of 16-column chunks, 128 / 256-column tiles
    plus the last column; k cycling through `ks` (default: the first and last k, the last full k-block's last k and
    the ragged block's first).  Sorted rows are paired with the reversed columns."""
    rows = sorted({i for i in (0, 31, 32, 127, 128, 255, 256, M - 33, M - 32, M - 1) if 0 <= i < M})
    cols = sorted({j for j in (0, 15, 16, 127, 128, 255, 256, 511, 512, N - 17, N - 16, N - 1) if 0 <= j < N})
    if ks is None:
        ks = [0, K - 1, (K - 1) // BK * BK, (K - 1) // BK * BK - 1]
    ks = [k for k in ks if 0 <= k < K]
    n = min(len(rows), len(cols))
    return [(rows[t], cols[::-1][t], ks[t % len(ks)]) for t in range(n)]


def split_hi_lo(x):
    """fp32 -> (bf16 hi, bf16 lo) with hi + lo ~= x to 2^-16 (what hba_split_bf16 writes)."""
    hi = x.to(torch.bfloat16)
    return hi, (x - hi.float()).to(torch.bfloat16)
