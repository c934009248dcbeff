"""ORACLE (test infrastructure only; nothing under vit-project_b200/ imports this, and the product has no switch
that routes to it: `import hba` needs the compiled libhba.so and every front end refuses non-CUDA tensors).

A CPU restatement of the C-ABI of include/hba.h, entry point by entry point, following the contracts written in the
header (which cite the reference lines each entry replaces): the same pointer / leading-dimension / hi-lo operand
conventions, computed with torch on host memory.  `RefLib` has the method names of the shared library, so that a test
can stand it in for `hba._lib.load()` and run the host side of the product - hba/ops.py, hba/engine.py (forward,
live-sub-graph backward, trunk cache), hba/dora.py, hba/optim.py, hba/rsa.py and the drop-in pipelines - unmodified on
CPU tensors (`emulated_device()` below; tests/test_host_on_ref_lib_cpu.py).  What that checks is the SEQUENCING of the
C-ABI calls (which buffers feed which call, the graph pruning, the cache, the fused-loss / NaN-guard / optimiser
wiring), against the oracle model and against the reference's own pipeline executed on the CPU.  It says nothing about
the CUDA kernels - those are compared with their formulas on a B200 by the `-m gpu` tests.

Every entry point of the header is restated (CLIP path and ViT-B/16 path).  The restatement is pinned by the GPU op
tests themselves: tests/emulate_clip_gpu_tests.py runs tests/test_gpu_ops.py on it, i.e. each restated entry point is
compared with the same torch / fp64-autograd / numpy / scipy formulas that judge the CUDA kernels.  The argument
checks of the front ends (HBA_REQUIRE) are restated as well; not restated: anything about scheduling (split-K order,
max_ctas, workspace use).

Arithmetic notes: GEMMs accumulate hi.hi + lo.hi + hi.lo in fp32 like the kernel (nsplit = 3) or the plain bf16 product
(nsplit = 1); attention keeps P in fp32 (the tensor-core kernel rounds P to bf16); everything else is the header's
formula in fp32 / fp64.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import math
import os

import numpy as np
import torch

_SIZE = {torch.float32: 4, torch.bfloat16: 2, torch.float64: 8, torch.int64: 8, torch.int32: 4, torch.uint8: 1}
DT = {0: torch.float32, 1: torch.bfloat16}


def _addr(p):
    if p is None:
        return 0
    if isinstance(p, C.c_void_p):
        return p.value or 0
    return int(p)


def flat(p, n, dtype):
    """n elements of `dtype` at address p as a torch tensor sharing the memory."""
    a = _addr(p)
    if a == 0:
        return None
    buf = (C.c_char * (n * _SIZE[dtype])).from_address(a)
    return torch.frombuffer(buf, dtype=dtype, count=n)


def mat(p, rows, cols, ld, dtype):
    """[rows, cols] view with row stride ld (elements)."""
    if _addr(p) == 0:
        return None
    if rows == 0:
        return torch.empty(0, cols, dtype=dtype)
    return flat(p, (rows - 1) * ld + cols, dtype).as_strided((rows, cols), (ld, 1))


def read_operand(p, rows, cols, ld, lo_off, parts=False):
    """bf16 hi[/lo] operand -> fp32 value (or the (hi, lo) pair)."""
    hi = mat(p, rows, cols, ld, torch.bfloat16).float()
    lo = None
    if lo_off > 0:
        lo = flat(p, (rows - 1) * ld + lo_off + cols, torch.bfloat16).as_strided((rows, cols), (ld, 1), lo_off).float()
    if parts:
        return hi, lo
    return hi if lo is None else hi + lo


def write_operand(p, value, ld, lo_off):
    rows, cols = value.shape
    hi = value.to(torch.bfloat16)
    mat(p, rows, cols, ld, torch.bfloat16).copy_(hi)
    if lo_off > 0:
        lo = (value - hi.float()).to(torch.bfloat16)
        flat(p, (rows - 1) * ld + lo_off + cols, torch.bfloat16).as_strided((rows, cols), (ld, 1), lo_off).copy_(lo)


def _act(v, act, aux):
    if act == 0:
        return v
    if act == 1:                                   # QuickGELU: x * sigmoid(1.702 x)
        return v * torch.sigmoid(1.702 * v)
    if act == 2:                                   # erf-GELU (torch's fp32 CPU gelu is off by ~1e-3 near -3.5)
        return torch.nn.functional.gelu(v.double()).to(v.dtype)
    a = aux.float()
    if act == 3:                                   # v * QuickGELU'(aux)
        s = torch.sigmoid(1.702 * a)
        return v * (s + 1.702 * a * s * (1 - s))
    if act == 4:
        cdf = 0.5 * (1 + torch.erf(a / math.sqrt(2.0)))
        pdf = torch.exp(-0.5 * a * a) / math.sqrt(2 * math.pi)
        return v * (cdf + a * pdf)
    raise ValueError(act)


class _ArgError(Exception):
    pass


def _require(cond, msg):
    if not cond:
        raise _ArgError(msg)


def _al(p, n=16):
    return _addr(p) % n == 0


HBA_ERR_ARG = -22


class RefLib:
    """Method-for-method stand-in of libhba.so on host memory (see the module docstring).  The argument checks of the
    library's front ends (HBA_REQUIRE: null pointers, shape limits, leading-dimension and 16-byte pointer alignment
    rules of the vectorised / TMA accesses) are restated too and answer like the library: HBA_ERR_ARG and a message
    in hba_last_error() - so a host-side call that the device would refuse is refused here as well."""

    def __init__(self):
        self.calls = []            # entry-point names in call order (tests assert on the sequencing)
        self._err = b""

    def __getattribute__(self, name):
        fn = object.__getattribute__(self, name)
        if not name.startswith("hba_") or name in ("hba_last_error", "hba_abi_version", "hba_device_check",
                                                   "hba_rank_workspace_bytes"):
            return fn

        def guarded(*args):
            try:
                return fn(*args)
            except _ArgError as exc:
                object.__setattr__(self, "_err", f"{name}: {exc}".encode())
                return HBA_ERR_ARG
        return guarded

    # ---------------------------------------------------------------- plumbing
    def hba_last_error(self):
        return self._err

    def hba_abi_version(self):
        return 1

    def hba_device_check(self):
        return 0

    def _ok(self, name):
        self.calls.append(name)
        return 0

    # ---------------------------------------------------------------- GEMM
    def hba_gemm_bf16(self, pref, stream):
        p = pref._obj if hasattr(pref, "_obj") else pref
        M, N, K = p.M, p.N, p.K
        _require(p.A and p.B, "null operand")
        _require(M > 0 and N > 0 and K > 0, f"empty problem M={M} N={N} K={K}")
        _require(p.lda % 8 == 0 and p.ldb % 8 == 0, "lda/ldb must be multiples of 8")
        _require(_al(p.A) and _al(p.B), "TMA operand must be 16-byte aligned")
        _require(p.nsplit in (1, 3), "nsplit must be 1 or 3")
        kpad = (K + 63) // 64 * 64
        if p.nsplit == 3:
            _require(p.a_lo_off >= (M if p.a_mn_major else kpad) and p.b_lo_off >= (N if p.b_mn_major else kpad)
                     and p.a_lo_off % 8 == 0 and p.b_lo_off % 8 == 0,
                     "lo offsets must lie behind the hi part and be multiples of 8")
        _require(p.out_f32 or p.out_bf16 or p.pre_out, "no output")
        _require(0 <= p.act <= 4, "bad act")
        if p.act in (3, 4):
            _require(p.aux, "activation gradient needs aux")
            _require(p.ld_aux % 4 != 0 or _al(p.aux, 16 if p.aux_dtype == 0 else 8),
                     "aux with ld % 4 == 0 must be 16-byte (f32) / 8-byte (bf16) aligned")
        if p.transpose_out:
            _require(p.act == 0 and not p.residual and not p.pre_out, "transpose_out supports alpha and bias only")
        else:
            _require(not p.out_f32 or (p.ld_f32 % 4 == 0 and _al(p.out_f32)), "out_f32 must be 16-byte aligned with ld % 4 == 0")
            _require(not p.out_bf16 or (p.ld_bf16 % 8 == 0 and p.out_lo_off % 8 == 0 and _al(p.out_bf16)),
                     "out_bf16 must be 16-byte aligned with ld % 8 == 0")
        _require(not p.residual or (p.ldr % 4 == 0 and _al(p.residual)), "residual must be 16-byte aligned with ld % 4 == 0")
        _require(not p.bias or _al(p.bias), "bias must be 16-byte aligned")
        if p.pre_out:
            _require(_al(p.pre_out) and p.ld_pre % 8 == 0, "pre_out must be 16-byte aligned with ld % 8 == 0")
        if p.colsum_partial:
            _require(p.out_bf16 and not p.transpose_out and N % 4 == 0 and _al(p.colsum_partial),
                     "colsum_partial needs a bf16 output, N % 4 == 0 and a 16-byte aligned buffer")
        if min(p.k_slices, (K + 63) // 64) > 1:
            _require(p.k_workspace and not p.transpose_out and not p.colsum_partial and N % 4 == 0,
                     f"split-K (k_slices={p.k_slices}) needs k_workspace, N % 4 == 0 and no transposed / column-sum output")
            _require(_al(p.k_workspace), "k_workspace must be 16-byte aligned")
        split = p.nsplit == 3

        def operand(ptr, ld, lo_off, rows, mn):
            if mn:      # stored [K, rows] (MN-major)
                hi, lo = read_operand(ptr, K, rows, ld, lo_off if split else 0, parts=True)
                return hi.t(), (lo.t() if lo is not None else None)
            return read_operand(ptr, rows, K, ld, lo_off if split else 0, parts=True)
        ah, al = operand(p.A, p.lda, p.a_lo_off, M, p.a_mn_major)
        bh, bl = operand(p.B, p.ldb, p.b_lo_off, N, p.b_mn_major)
        acc = ah @ bh.t()
        if split:
            acc = acc + al @ bh.t() + ah @ bl.t()
        v = p.alpha * acc
        if p.bias:
            v = v + flat(p.bias, N, torch.float32)
        if p.transpose_out:
            vt = v.t().contiguous()
            if p.out_f32:
                mat(p.out_f32, N, M, p.ld_f32, torch.float32).copy_(vt)
            if p.out_bf16:
                write_operand(p.out_bf16, vt, p.ld_bf16, p.out_lo_off)
            return self._ok("hba_gemm_bf16")
        if p.pre_out:
            mat(p.pre_out, M, N, p.ld_pre, DT[p.pre_dtype]).copy_(v.to(DT[p.pre_dtype]))
        aux = mat(p.aux, M, N, p.ld_aux, DT[p.aux_dtype]) if p.aux else None
        v = _act(v, p.act, aux)
        if p.residual:
            v = v + mat(p.residual, M, N, p.ldr, torch.float32)
        if p.out_f32:
            mat(p.out_f32, M, N, p.ld_f32, torch.float32).copy_(v)
        if p.out_bf16:
            write_operand(p.out_bf16, v, p.ld_bf16, p.out_lo_off)
        if p.colsum_partial:
            hi = v.to(torch.bfloat16).float()
            groups = (M + 31) // 32
            out = flat(p.colsum_partial, groups * N, torch.float32).view(groups, N)
            for g in range(groups):
                out[g] = hi[32 * g:32 * g + 32].sum(0)
        return self._ok("hba_gemm_bf16")

    def hba_split_bf16(self, x, rows, cols, ld_in, out, ld_out, lo_off, transpose, stream):
        _require(_addr(x) and _addr(out) and rows > 0 and cols > 0, "bad arguments")
        if not transpose:
            _require(cols % 4 == 0 and ld_in % 4 == 0 and ld_out % 2 == 0 and lo_off % 2 == 0 and _al(x) and _al(out, 4),
                     "cols/ld must be multiples of 4 and pointers aligned")
        v = mat(x, rows, cols, ld_in, torch.float32)
        write_operand(out, v.t().contiguous() if transpose else v, ld_out, lo_off)
        return self._ok("hba_split_bf16")

    # ---------------------------------------------------------------- LayerNorm
    @staticmethod
    def _rows(p, rows, cols, ld, step):
        return flat(p, ((rows - 1) * step) * ld + cols, torch.float32).as_strided((rows, cols), (ld * step, 1))

    def hba_layernorm_fwd(self, x, rows, cols, ldx, row_step, gamma, beta, eps, y_f32, ld_yf, y_bf16, ld_yb, lo_off,
                          stream):
        _require(_addr(x) and _addr(gamma) and _addr(beta) and (_addr(y_f32) or _addr(y_bf16)) and rows > 0, "bad arguments")
        _require(cols % 128 == 0 and cols <= 1024, f"cols={cols} must be a multiple of 128 and <= 1024")
        _require(ldx % 4 == 0 and ld_yf % 4 == 0 and ld_yb % 4 == 0 and lo_off % 4 == 0 and _al(y_bf16, 8),
                 "leading dimensions must keep 16-byte (fp32) / 8-byte (bf16) row alignment")
        _require(_al(x) and _al(gamma) and _al(beta) and _al(y_f32), "x, gamma, beta and y_f32 must be 16-byte aligned")
        row_step = max(1, row_step)
        xv = self._rows(x, rows, cols, ldx, row_step)
        mu = xv.mean(1, keepdim=True)
        var = ((xv - mu) ** 2).mean(1, keepdim=True)
        y = (xv - mu) / torch.sqrt(var + eps) * flat(gamma, cols, torch.float32) + flat(beta, cols, torch.float32)
        if _addr(y_f32):
            mat(y_f32, rows, cols, ld_yf, torch.float32).copy_(y)
        if _addr(y_bf16):
            write_operand(y_bf16, y, ld_yb, lo_off)
        return self._ok("hba_layernorm_fwd")

    def hba_layernorm_bwd(self, dy, ld_dy, x, rows, cols, ldx, row_step, gamma, eps, dx, ld_dx, accumulate, stream):
        _require(_addr(dy) and _addr(x) and _addr(gamma) and _addr(dx) and rows > 0, "bad arguments")
        _require(cols % 128 == 0 and cols <= 1024, f"cols={cols} must be a multiple of 128 and <= 1024")
        _require(ldx % 4 == 0 and ld_dy % 4 == 0 and ld_dx % 4 == 0, "leading dimensions must be multiples of 4")
        _require(_al(dy) and _al(x) and _al(gamma) and _al(dx), "dy, x, gamma and dx must be 16-byte aligned")
        row_step = max(1, row_step)
        xv = self._rows(x, rows, cols, ldx, row_step)
        g = mat(dy, rows, cols, ld_dy, torch.float32) * flat(gamma, cols, torch.float32)
        mu = xv.mean(1, keepdim=True)
        rstd = 1.0 / torch.sqrt(((xv - mu) ** 2).mean(1, keepdim=True) + eps)
        xhat = (xv - mu) * rstd
        d = rstd * (g - g.mean(1, keepdim=True) - xhat * (g * xhat).mean(1, keepdim=True))
        out = mat(dx, rows, cols, ld_dx, torch.float32)
        out.copy_(out + d if accumulate else d)
        return self._ok("hba_layernorm_bwd")

    # ---------------------------------------------------------------- front ends of the towers
    def hba_im2col_patches(self, image, B, H, W, P, out, ld_out, lo_off, stream):
        _require(_addr(image) and _addr(out) and B > 0 and P > 0 and H % P == 0 and W % P == 0, "bad arguments")
        _require((ld_out if lo_off == 0 else lo_off) >= 3 * P * P and (lo_off == 0 or ld_out - lo_off >= 3 * P * P),
                 "row too short for 3*P*P columns")
        img = flat(image, B * 3 * H * W, torch.float32).view(B, 3, H, W)
        gh, gw = H // P, W // P
        cols = img.view(B, 3, gh, P, gw, P).permute(0, 2, 4, 1, 3, 5).reshape(B * gh * gw, 3 * P * P)
        # zeros up to lo_off in the hi part (up to ld_out without a lo part) and up to ld_out in the lo part
        padded = torch.zeros(B * gh * gw, lo_off if lo_off > 0 else ld_out)
        padded[:, :3 * P * P] = cols
        write_operand(out, padded, ld_out, 0)
        if lo_off > 0:
            lo = torch.zeros(B * gh * gw, ld_out - lo_off)
            lo[:, :3 * P * P] = cols - cols.to(torch.bfloat16).float()
            write_operand(_addr(out) + 2 * lo_off, lo, ld_out, 0)
        return self._ok("hba_im2col_patches")

    def hba_assemble_tokens_ln(self, conv, B, n_patches, width, cls, pos, gamma, beta, eps, x_out, stream):
        _require(_addr(conv) and _addr(cls) and _addr(pos) and _addr(x_out) and B > 0 and (not _addr(gamma)) == (not _addr(beta)),
                 "bad arguments")
        _require(width % 128 == 0 and width <= 1024, f"width={width} unsupported")
        _require(all(_al(p) for p in (conv, cls, pos, gamma, beta, x_out)),
                 "conv, cls, pos, gamma, beta and x_out must be 16-byte aligned")
        c = flat(conv, B * n_patches * width, torch.float32).view(B, n_patches, width)
        ps = flat(pos, (n_patches + 1) * width, torch.float32).view(n_patches + 1, width)
        x = torch.cat([flat(cls, width, torch.float32).expand(B, 1, width), c], 1) + ps
        if _addr(gamma):
            x = torch.nn.functional.layer_norm(x, (width,), flat(gamma, width, torch.float32),
                                               flat(beta, width, torch.float32), eps)
        flat(x_out, B * (n_patches + 1) * width, torch.float32).copy_(x.reshape(-1))
        return self._ok("hba_assemble_tokens_ln")

    def hba_embed_tokens(self, tokens, S, T, width, table, pos, x_out, stream):
        _require(_addr(tokens) and _addr(table) and _addr(pos) and _addr(x_out) and S > 0 and T > 0 and width % 4 == 0,
                 "bad arguments")
        _require(_al(table) and _al(pos) and _al(x_out), "table, pos and x_out must be 16-byte aligned")
        tok = flat(tokens, S * T, torch.int64).view(S, T)
        n_vocab = int(tok.max()) + 1
        tab = flat(table, n_vocab * width, torch.float32).view(n_vocab, width)
        x = tab[tok] + flat(pos, T * width, torch.float32).view(T, width)
        flat(x_out, S * T * width, torch.float32).copy_(x.reshape(-1))
        return self._ok("hba_embed_tokens")

    def hba_gather_rows(self, src, ld_in, idx, n, cols, out, ld_out, stream):
        _require(_addr(src) and _addr(idx) and _addr(out) and n > 0 and cols > 0, "bad arguments")
        ix = flat(idx, n, torch.int64)
        rows = int(ix.max()) + 1
        mat(out, n, cols, ld_out, torch.float32).copy_(mat(src, rows, cols, ld_in, torch.float32)[ix])
        return self._ok("hba_gather_rows")

    # ---------------------------------------------------------------- attention
    @staticmethod
    def _qkv(qkv, dtype, ld, B, T, H):
        m = mat(qkv, B * T, 3 * H * 64, ld, DT[dtype]).float()
        q, k, v = (m[:, i * H * 64:(i + 1) * H * 64].reshape(B, T, H, 64).permute(0, 2, 1, 3) for i in range(3))
        return q, k, v       # [B, H, T, 64]

    def hba_attention_fwd(self, qkv, dtype, ld_qkv, B, T, H, causal, first_row_only, out, ld_out, lo_off, out_f32,
                          ld_of, stream):
        _require(_addr(qkv) and (_addr(out) or _addr(out_f32)) and B > 0 and T > 0 and H > 0, "bad arguments")
        _require(T <= 288, f"T={T} exceeds 288")
        _require(not (first_row_only and causal), "first_row_only with causal is unsupported")
        if first_row_only:
            _require(ld_qkv % 8 == 0 and _al(qkv), "first_row_only needs 16-byte aligned qkv rows (ld % 8 == 0)")
        _require(dtype in DT, f"unknown dtype {dtype}")
        q, k, v = self._qkv(qkv, dtype, ld_qkv, B, T, H)
        if first_row_only:
            q = q[:, :, :1]
        s = q @ k.transpose(-1, -2) / 8.0
        if causal:
            Tq = s.shape[-2]
            s = s.masked_fill(torch.ones(Tq, T, dtype=torch.bool).triu(1), float("-inf"))
        o = (torch.softmax(s, -1) @ v).permute(0, 2, 1, 3).reshape(-1, H * 64)
        if _addr(out):
            write_operand(out, o, ld_out, lo_off)
        if _addr(out_f32):
            mat(out_f32, o.shape[0], H * 64, ld_of, torch.float32).copy_(o)
        return self._ok("hba_attention_fwd")

    def hba_attention_bwd_row0(self, qkv, dtype, ld_qkv, B, T, H, d_out, ld_do, d_qkv, ld_dqkv, stream):
        _require(_addr(qkv) and _addr(d_out) and _addr(d_qkv) and B > 0 and T > 0 and H > 0, "bad arguments")
        _require(T <= 288, f"T={T} exceeds 288")
        _require(ld_qkv % 8 == 0 and _al(qkv) and ld_dqkv % 4 == 0 and _al(d_qkv), "qkv / d_qkv rows must be 16-byte aligned")
        q, k, v = self._qkv(qkv, dtype, ld_qkv, B, T, H)
        q0 = q[:, :, :1]                                                     # [B, H, 1, 64]
        p = torch.softmax(q0 @ k.transpose(-1, -2) / 8.0, -1)               # [B, H, 1, T]
        do = mat(d_out, B, H * 64, ld_do, torch.float32).view(B, H, 1, 64)
        dv = p.transpose(-1, -2) @ do                                        # [B, H, T, 64]
        dp = do @ v.transpose(-1, -2)                                        # [B, H, 1, T]
        ds = p * (dp - (dp * p).sum(-1, keepdim=True)) / 8.0
        dq0 = ds @ k                                                         # [B, H, 1, 64]
        dk = ds.transpose(-1, -2) @ q0                                       # [B, H, T, 64]
        dq = torch.zeros(B, H, T, 64)
        dq[:, :, :1] = dq0
        full = torch.cat([t.permute(0, 2, 1, 3).reshape(B * T, H * 64) for t in (dq, dk, dv)], 1)
        mat(d_qkv, B * T, 3 * H * 64, ld_dqkv, torch.float32).copy_(full)
        return self._ok("hba_attention_bwd_row0")

    # ---------------------------------------------------------------- DoRA (NEW:447-463 and its autograd)
    def hba_dora_merge_fwd(self, D, A, Bm, m, in_f, out_f, r, scale, eps, w_t_f32, w_bf16, ld_w, w_lo_off, wt_bf16,
                           ld_wt, wt_lo_off, norm_out, stream):
        _require(_addr(D) and _addr(A) and _addr(Bm) and _addr(m), "null input")
        _require(_addr(w_t_f32) or _addr(w_bf16) or _addr(wt_bf16), "no output requested")
        self._dora_check(in_f, out_f, r)
        _require(not _addr(wt_bf16) or (ld_wt % 8 == 0 and wt_lo_off % 8 == 0 and _al(wt_bf16)), "wt_bf16 alignment")
        Dv = flat(D, in_f * out_f, torch.float32).view(in_f, out_f)
        V = Dv + scale * (flat(Bm, in_f * r, torch.float32).view(in_f, r) @ flat(A, r * out_f, torch.float32).view(r, out_f))
        n = torch.norm(V, dim=0) + eps
        Wt = V / n * flat(m, out_f, torch.float32)
        if _addr(w_t_f32):
            flat(w_t_f32, in_f * out_f, torch.float32).copy_(Wt.reshape(-1))
        if _addr(w_bf16):
            write_operand(w_bf16, Wt.t().contiguous(), ld_w, w_lo_off)
        if _addr(wt_bf16):
            write_operand(wt_bf16, Wt.contiguous(), ld_wt, wt_lo_off)
        if _addr(norm_out):
            flat(norm_out, out_f, torch.float32).copy_(n)
        return self._ok("hba_dora_merge_fwd")

    @staticmethod
    def _dora_check(in_f, out_f, r):
        _require(0 < in_f <= 2048, f"in_features={in_f} unsupported (max 2048)")
        _require(out_f > 0 and out_f % 8 == 0, f"out_features={out_f} must be a multiple of 8")
        _require(0 < r <= 64 and r % 4 == 0, f"rank={r} must be a multiple of 4 and <= 64")

    def hba_dora_merge_bwd(self, G, ld_g, D, A, Bm, m, in_f, out_f, r, scale, eps, dm, dA, dB, workspace, stream):
        _require(all(_addr(t) for t in (G, D, A, Bm, m, dm, dA, dB, workspace)), "null pointer")
        self._dora_check(in_f, out_f, r)
        _require(out_f <= 1792, f"out_features={out_f} exceeds the shared-memory staging (max 1792)")
        Gt = mat(G, out_f, in_f, ld_g, torch.float32).t()                   # dL/dWt [in, out]
        Dv = flat(D, in_f * out_f, torch.float32).view(in_f, out_f)
        Av = flat(A, r * out_f, torch.float32).view(r, out_f)
        Bv = flat(Bm, in_f * r, torch.float32).view(in_f, r)
        mv = flat(m, out_f, torch.float32)
        V = Dv + scale * (Bv @ Av)
        nv = torch.norm(V, dim=0)
        n = nv + eps
        gv = (Gt * V).sum(0)
        flat(dm, out_f, torch.float32).copy_(gv / n)
        dV = (mv / n) * (Gt - V * gv / (n * nv))
        flat(dA, r * out_f, torch.float32).copy_((scale * (Bv.t() @ dV)).reshape(-1))
        flat(dB, in_f * r, torch.float32).copy_((scale * (dV @ Av.t())).reshape(-1))
        return self._ok("hba_dora_merge_bwd")

    # ---------------------------------------------------------------- cosine head (+ MSE)
    @staticmethod
    def _cos(img, txt, logit_scale):
        ni, nt = img.norm(dim=1, keepdim=True), txt.norm(dim=1, keepdim=True)
        s = torch.exp(logit_scale)
        return s * (img / ni) @ (txt / nt).t(), ni, nt, s

    def hba_cos_head_fwd(self, img, txt, B, Cn, E, logit_scale, pred, target, loss, stream):
        _require(_addr(img) and _addr(txt) and _addr(logit_scale) and _addr(pred) and B > 0 and Cn > 0, "bad arguments")
        _require(E > 0 and E % 4 == 0, f"E={E} must be a multiple of 4")
        _require(not _addr(loss) or _addr(target), "loss requested without target")
        pr, *_ = self._cos(flat(img, B * E, torch.float32).view(B, E), flat(txt, Cn * E, torch.float32).view(Cn, E),
                           flat(logit_scale, 1, torch.float32))
        flat(pred, B * Cn, torch.float32).copy_(pr.reshape(-1))
        if _addr(target) and _addr(loss):
            flat(loss, 1, torch.float32).copy_(((pr - flat(target, B * Cn, torch.float32).view(B, Cn)) ** 2).mean().reshape(1))
        return self._ok("hba_cos_head_fwd")

    def _cos_bwd(self, img, txt, logit_scale, dp):
        pr, ni, nt, s = self._cos(img, txt, logit_scale)
        ih, th = img / ni, txt / nt
        g_ih = s * dp @ th
        g_th = s * dp.t() @ ih
        d_img = (g_ih - ih * (g_ih * ih).sum(1, keepdim=True)) / ni
        d_txt = (g_th - th * (g_th * th).sum(1, keepdim=True)) / nt
        return d_img, d_txt

    def hba_cos_head_bwd(self, img, txt, B, Cn, E, logit_scale, d_pred, pred, target, d_img, d_txt, stream):
        _require(_addr(img) and _addr(txt) and _addr(logit_scale) and (_addr(d_img) or _addr(d_txt)) and B > 0 and Cn > 0,
                 "bad arguments")
        _require(_addr(d_pred) or (_addr(pred) and _addr(target)), "need d_pred or (pred, target)")
        _require(E % 4 == 0 and E <= 2048, f"E={E} unsupported")
        _require(B <= 1024 and Cn <= 1024, "B, C must be <= 1024")
        iv, tv = flat(img, B * E, torch.float32).view(B, E), flat(txt, Cn * E, torch.float32).view(Cn, E)
        if _addr(d_pred):
            dp = flat(d_pred, B * Cn, torch.float32).view(B, Cn)
        else:
            dp = 2.0 * (flat(pred, B * Cn, torch.float32) - flat(target, B * Cn, torch.float32)).view(B, Cn) / (B * Cn)
        di, dt = self._cos_bwd(iv, tv, flat(logit_scale, 1, torch.float32), dp)
        flat(d_img, B * E, torch.float32).copy_(di.reshape(-1))
        flat(d_txt, Cn * E, torch.float32).copy_(dt.reshape(-1))
        return self._ok("hba_cos_head_bwd")

    def hba_cos_mse_fwd(self, img, txt, B, Cn, E, groups, logit_scale, pred, target, tstride, loss, bad_step,
                        bad_total, total, workspace, stream):
        _require(_addr(img) and _addr(txt) and _addr(logit_scale) and _addr(pred) and B > 0 and Cn > 0 and groups > 0,
                 "bad arguments")
        _require(E > 0 and E % 4 == 0, f"E={E} must be a multiple of 4")
        _require(groups <= 65535, "too many groups")
        if _addr(target):
            _require(_addr(loss) and _addr(workspace), "target given without loss / workspace")
        else:
            _require(not (_addr(loss) or _addr(bad_step) or _addr(bad_total) or _addr(total)),
                     "loss outputs requested without target")
        ls = flat(logit_scale, 1, torch.float32)
        for g in range(groups):
            iv = flat(_addr(img) + 4 * g * B * E, B * E, torch.float32).view(B, E)
            tv = flat(_addr(txt) + 4 * g * Cn * E, Cn * E, torch.float32).view(Cn, E)
            pr, *_ = self._cos(iv, tv, ls)
            flat(_addr(pred) + 4 * g * B * Cn, B * Cn, torch.float32).copy_(pr.reshape(-1))
            if not _addr(target):
                continue
            tg = flat(_addr(target) + 4 * g * tstride, B * Cn, torch.float32).view(B, Cn)
            l = ((pr - tg) ** 2).mean()
            flat(loss, groups, torch.float32)[g] = l
            bad = int(not bool(torch.isfinite(l)))
            if _addr(bad_step):
                flat(bad_step, groups, torch.int32)[g] = bad
            if _addr(bad_total):
                flat(bad_total, groups, torch.int32)[g] += bad if _addr(bad_step) else 0
            if _addr(total) and not (bad and _addr(bad_step)):
                flat(total, groups, torch.float64)[g] += float(l) * B
        return self._ok("hba_cos_mse_fwd")

    def hba_cos_mse_bwd(self, img, txt, B, Cn, E, groups, logit_scale, pred, target, tstride, d_loss, d_img, d_txt,
                        stream):
        _require(_addr(img) and _addr(txt) and _addr(logit_scale) and _addr(pred) and _addr(target)
                 and (_addr(d_img) or _addr(d_txt)) and B > 0 and Cn > 0 and groups > 0, "bad arguments")
        _require(E % 4 == 0 and E <= 2048, f"E={E} unsupported")
        _require(B <= 1024 and Cn <= 1024 and groups <= 65535, "B, C must be <= 1024")
        ls = flat(logit_scale, 1, torch.float32)
        for g in range(groups):
            iv = flat(_addr(img) + 4 * g * B * E, B * E, torch.float32).view(B, E)
            tv = flat(_addr(txt) + 4 * g * Cn * E, Cn * E, torch.float32).view(Cn, E)
            pr = flat(_addr(pred) + 4 * g * B * Cn, B * Cn, torch.float32).view(B, Cn)
            tg = flat(_addr(target) + 4 * g * tstride, B * Cn, torch.float32).view(B, Cn)
            up = float(flat(d_loss, groups, torch.float32)[g]) if _addr(d_loss) else 1.0
            di, dt = self._cos_bwd(iv, tv, ls, 2.0 * (pr - tg) / (B * Cn) * up)
            flat(_addr(d_img) + 4 * g * B * E, B * E, torch.float32).copy_(di.reshape(-1))
            flat(_addr(d_txt) + 4 * g * Cn * E, Cn * E, torch.float32).copy_(dt.reshape(-1))
        return self._ok("hba_cos_mse_bwd")

    # ---------------------------------------------------------------- AdamW (torch.optim.AdamW arithmetic, NEW:1181)
    def hba_adamw_multi(self, ptrs, sizes, n, total, lr, beta1, beta2, eps, weight_decay, step, step_dev, skip_flag,
                        stream):
        _require(_addr(ptrs) and _addr(sizes) and 0 < n <= 1024 and total > 0 and (step >= 1 or _addr(step_dev)),
                 "bad arguments")
        if _addr(skip_flag) and int(flat(skip_flag, 1, torch.int32)[0]) != 0:
            return self._ok("hba_adamw_multi")
        if _addr(step_dev):
            step = int(flat(step_dev, 1, torch.int32)[0])
        table = flat(ptrs, 4 * n, torch.int64).view(n, 4)
        sz = flat(sizes, n, torch.int64)
        bc1, bc2 = 1 - beta1 ** step, 1 - beta2 ** step
        for i in range(n):
            k = int(sz[i])
            p, g, m, v = (flat(int(table[i, j]), k, torch.float32) for j in range(4))
            p.mul_(1 - lr * weight_decay)
            m.mul_(beta1).add_(g, alpha=1 - beta1)
            v.mul_(beta2).addcmul_(g, g, value=1 - beta2)
            p.addcdiv_(m, v.sqrt() / math.sqrt(bc2) + eps, value=-lr / bc1)
        return self._ok("hba_adamw_multi")

    def hba_sgd_multi(self, ptrs, sizes, n, total, lr, momentum, weight_decay, first_step, skip_flag, stream):
        """torch.optim.SGD(momentum, weight_decay, dampening 0, no nesterov), VIT:294-299."""
        if _addr(skip_flag) and int(flat(skip_flag, 1, torch.int32)[0]) != 0:
            return self._ok("hba_sgd_multi")
        table = flat(ptrs, 3 * n, torch.int64).view(n, 3)
        sz = flat(sizes, n, torch.int64)
        for i in range(n):
            k = int(sz[i])
            p, g, buf = (flat(int(table[i, j]), k, torch.float32) for j in range(3))
            d = g + weight_decay * p
            if first_step:
                buf.copy_(d)
            else:
                buf.mul_(momentum).add_(d)
            p.add_(buf, alpha=-lr)
        return self._ok("hba_sgd_multi")

    def hba_sgd_staged(self, ptrs, prefix4, n, total4, lr, momentum, weight_decay, first_step, skip_flag, stream):
        if _addr(skip_flag) and int(flat(skip_flag, 1, torch.int32)[0]) != 0:
            return self._ok("hba_sgd_staged")
        table = flat(ptrs, 4 * n, torch.int64).view(n, 4)
        pre = flat(prefix4, n, torch.int64).tolist() + [int(total4)]
        for i in range(n):
            k = 4 * (pre[i + 1] - pre[i])
            p, g, buf = (flat(int(table[i, j]), k, torch.float32) for j in range(3))
            d = g + weight_decay * p
            if first_step:
                buf.copy_(d)
            else:
                buf.mul_(momentum).add_(d)
            p.add_(buf, alpha=-lr)
            if int(table[i, 3]):
                flat(int(table[i, 3]), k, torch.bfloat16).copy_(p.to(torch.bfloat16))
        return self._ok("hba_sgd_staged")

    # ---------------------------------------------------------------- ViT-B/16 training step (VIT:125-165)
    def hba_softmax_ce_fwd_bwd(self, logits, ld, labels, B, Cn, loss, d_logits, ld_d, correct, workspace, stream):
        z = mat(logits, B, Cn, ld, torch.float32)
        y = flat(labels, B, torch.int64)
        logp = torch.log_softmax(z, 1)
        flat(loss, 1, torch.float32)[0] = -logp[torch.arange(B), y].mean()
        if _addr(d_logits):
            d = torch.softmax(z, 1)
            d[torch.arange(B), y] -= 1
            mat(d_logits, B, Cn, ld_d, torch.float32).copy_(d / B)
        if _addr(correct):
            flat(correct, 1, torch.int32)[0] = int((z.argmax(1) == y).sum())
        return self._ok("hba_softmax_ce_fwd_bwd")

    def hba_colsum(self, x, dtype, rows, cols, ld, out, accumulate, workspace, stream):
        _require(_addr(x) and _addr(out) and _addr(workspace) and rows > 0 and cols > 0, "bad arguments")
        _require(dtype in DT, f"unknown dtype {dtype}")
        s_ = mat(x, rows, cols, ld, DT[dtype]).float().sum(0)
        o = flat(out, cols, torch.float32)
        o.copy_(o + s_ if accumulate else s_)
        return self._ok("hba_colsum")

    def _ln_stats(self, x, rows, cols, ldx, row_step, eps):
        xv = self._rows(x, rows, cols, ldx, row_step)
        mu = xv.mean(1, keepdim=True)
        rstd = 1.0 / torch.sqrt(((xv - mu) ** 2).mean(1, keepdim=True) + eps)
        return (xv - mu) * rstd, rstd

    def hba_layernorm_param_grad(self, dy, ld_dy, x, rows, cols, ldx, row_step, eps, dgamma_dbeta, accumulate,
                                 workspace, stream):
        _require(_addr(dy) and _addr(x) and _addr(dgamma_dbeta) and _addr(workspace) and rows > 0 and cols > 0
                 and cols % 4 == 0, "bad arguments")
        _require(ldx % 4 == 0 and _al(x), "x must be 16-byte aligned and ldx a multiple of 4")
        xhat, _ = self._ln_stats(x, rows, cols, ldx, max(1, row_step), eps)
        g = mat(dy, rows, cols, ld_dy, torch.float32)
        new = torch.cat([(g * xhat).sum(0), g.sum(0)])
        o = flat(dgamma_dbeta, 2 * cols, torch.float32)
        o.copy_(o + new if accumulate else new)
        return self._ok("hba_layernorm_param_grad")

    def hba_layernorm_bwd_fused(self, dy, ld_dy, x, rows, cols, ldx, gamma, eps, dx, ld_dx, accumulate, dx_bf16, ld_b,
                                lo_off, dgamma_dbeta, accumulate_params, dx_colsum, workspace, stream):
        _require(_addr(dy) and _addr(x) and _addr(gamma) and _addr(dx) and _addr(dgamma_dbeta) and _addr(workspace)
                 and rows > 0, "bad arguments")
        _require(ldx % 4 == 0 and ld_dy % 4 == 0 and ld_dx % 4 == 0 and ld_b % 4 == 0 and lo_off % 4 == 0,
                 "leading dimensions must be multiples of 4")
        _require(_al(dy) and _al(x) and _al(gamma) and _al(dx) and _al(dx_bf16, 8),
                 "dy, x, gamma and dx must be 16-byte aligned, dx_bf16 8-byte aligned")
        _require(cols in (128, 256, 512, 768, 1024), f"cols={cols} (supported: 128, 256, 512, 768, 1024)")
        xhat, rstd = self._ln_stats(x, rows, cols, ldx, 1, eps)
        g0 = mat(dy, rows, cols, ld_dy, torch.float32)
        g = g0 * flat(gamma, cols, torch.float32)
        d = rstd * (g - g.mean(1, keepdim=True) - xhat * (g * xhat).mean(1, keepdim=True))
        out = mat(dx, rows, cols, ld_dx, torch.float32)
        out.copy_(out + d if accumulate else d)
        if _addr(dx_bf16):
            write_operand(dx_bf16, out.clone(), ld_b, lo_off)
        new = torch.cat([(g0 * xhat).sum(0), g0.sum(0)])
        o = flat(dgamma_dbeta, 2 * cols, torch.float32)
        o.copy_(o + new if accumulate_params else new)
        if _addr(dx_colsum):
            flat(dx_colsum, cols, torch.float32).copy_(out.sum(0))
        return self._ok("hba_layernorm_bwd_fused")

    def _attn_bwd(self, q, k, v, do, causal):
        T = q.shape[2]
        s_ = q @ k.transpose(-1, -2) / 8.0
        if causal:
            s_ = s_.masked_fill(torch.ones(T, T, dtype=torch.bool).triu(1), float("-inf"))
        p = torch.softmax(s_, -1)
        dv = p.transpose(-1, -2) @ do
        dp = do @ v.transpose(-1, -2)
        ds = p * (dp - (dp * p).sum(-1, keepdim=True)) / 8.0
        return ds @ k, ds.transpose(-1, -2) @ q, dv

    def hba_attention_bwd(self, qkv, qkv_dtype, ld_qkv, B, T, H, causal, d_out, do_dtype, ld_do, d_qkv, dq_dtype,
                          ld_dqkv, stream):
        _require(_addr(qkv) and _addr(d_out) and _addr(d_qkv) and B > 0 and T > 0 and H > 0, "bad arguments")
        _require(T <= 288, f"T={T} exceeds 288")
        _require((qkv_dtype, do_dtype, dq_dtype) in ((1, 1, 1), (1, 0, 1), (0, 0, 0)),
                 f"unsupported dtype combination ({qkv_dtype}, {do_dtype}, {dq_dtype})")
        # (the fp32 form stages K / V / dK / dV of one head in shared memory: 4 * T * 64 floats + the per-warp rows)
        _require(qkv_dtype == 1 or T <= 200, f"fp32 form: T={T} exceeds the shared-memory staging (T <= 200)")
        q, k, v = self._qkv(qkv, qkv_dtype, ld_qkv, B, T, H)
        do = mat(d_out, B * T, H * 64, ld_do, DT[do_dtype]).float().reshape(B, T, H, 64).permute(0, 2, 1, 3)
        full = torch.cat([t.permute(0, 2, 1, 3).reshape(B * T, H * 64) for t in self._attn_bwd(q, k, v, do, causal)], 1)
        mat(d_qkv, B * T, 3 * H * 64, ld_dqkv, DT[dq_dtype]).copy_(full.to(DT[dq_dtype]))
        return self._ok("hba_attention_bwd")

    def hba_attention_fwd_lse(self, qkv, ld_qkv, B, T, H, causal, out, ld_out, lse, stream):
        _require(_addr(qkv) and _addr(out) and _addr(lse) and B > 0 and T > 0 and H > 0, "bad arguments")
        _require(T <= 257 and ld_qkv % 8 == 0 and ld_out % 8 == 0, f"T={T} (max 257) / leading dimensions unsupported")
        q, k, v = self._qkv(qkv, 1, ld_qkv, B, T, H)
        s_ = q @ k.transpose(-1, -2) / 8.0
        if causal:
            s_ = s_.masked_fill(torch.ones(T, T, dtype=torch.bool).triu(1), float("-inf"))
        o = (torch.softmax(s_, -1) @ v).permute(0, 2, 1, 3).reshape(B * T, H * 64)
        mat(out, B * T, H * 64, ld_out, torch.bfloat16).copy_(o.to(torch.bfloat16))
        flat(lse, B * H * T, torch.float32).copy_((torch.logsumexp(s_, -1) / math.log(2.0)).reshape(-1))
        return self._ok("hba_attention_fwd_lse")

    def hba_attention_bwd_lse(self, qkv, ld_qkv, B, T, H, causal, out, ld_out, d_out, ld_do, lse, d_qkv, ld_dqkv, stream):
        _require(_addr(qkv) and _addr(out) and _addr(d_out) and _addr(lse) and _addr(d_qkv) and B > 0 and T > 0 and H > 0,
                 "bad arguments")
        _require(T <= 256, f"T={T} exceeds 256")
        _require(ld_qkv % 8 == 0 and ld_out % 8 == 0 and ld_do % 8 == 0 and ld_dqkv % 8 == 0,
                 "leading dimensions must be multiples of 8")
        q, k, v = self._qkv(qkv, 1, ld_qkv, B, T, H)
        do = mat(d_out, B * T, H * 64, ld_do, torch.bfloat16).float().reshape(B, T, H, 64).permute(0, 2, 1, 3)
        full = torch.cat([t.permute(0, 2, 1, 3).reshape(B * T, H * 64) for t in self._attn_bwd(q, k, v, do, causal)], 1)
        mat(d_qkv, B * T, 3 * H * 64, ld_dqkv, torch.bfloat16).copy_(full.to(torch.bfloat16))
        return self._ok("hba_attention_bwd_lse")

    # ---------------------------------------------------------------- RSA tail (NEW:625-652)
    def hba_rdm_f64(self, E, N, Dm, rdm, tri, stream):
        e = flat(E, N * Dm, torch.float32).view(N, Dm).numpy().astype(np.float64)
        r = 1 - np.corrcoef(e)
        np.fill_diagonal(r, 0)
        if _addr(rdm):
            flat(rdm, N * N, torch.float64).copy_(torch.from_numpy(r.reshape(-1).copy()))
        if _addr(tri):
            flat(tri, N * (N - 1) // 2, torch.float64).copy_(torch.from_numpy(r[np.triu_indices(N, k=1)].copy()))
        return self._ok("hba_rdm_f64")

    def hba_rank_workspace_bytes(self, n):
        return 256 if n <= 2048 else 64 * int(n) + (1 << 20)

    def hba_rank_avg_f64(self, x, n, ranks, workspace, workspace_bytes, stream):
        from scipy.stats import rankdata
        flat(ranks, n, torch.float64).copy_(torch.from_numpy(rankdata(flat(x, n, torch.float64).numpy(), nan_policy="propagate")))
        return self._ok("hba_rank_avg_f64")

    def hba_pearson_f64(self, a, b, n, rho_out, workspace, stream):
        av, bv = flat(a, n, torch.float64).numpy(), flat(b, n, torch.float64).numpy()
        with np.errstate(all="ignore"):
            flat(rho_out, 1, torch.float64)[0] = float(np.corrcoef(av, bv)[0, 1])
        return self._ok("hba_pearson_f64")

    def hba_rdm_spearman(self, E, N, Dm, ref_ranks, rdm, ranks, rho_out, workspace, workspace_bytes, stream):
        from scipy.stats import rankdata
        P = N * (N - 1) // 2
        e = flat(E, N * Dm, torch.float32).view(N, Dm).numpy().astype(np.float64)
        with np.errstate(all="ignore"):
            r = 1 - np.corrcoef(e)
            np.fill_diagonal(r, 0)
            rk = rankdata(r[np.triu_indices(N, k=1)], nan_policy="propagate")
            flat(rho_out, 1, torch.float64)[0] = float(np.corrcoef(rk, flat(ref_ranks, P, torch.float64).numpy())[0, 1])
        if _addr(rdm):
            flat(rdm, N * N, torch.float64).copy_(torch.from_numpy(r.reshape(-1).copy()))
        if _addr(ranks):
            flat(ranks, P, torch.float64).copy_(torch.from_numpy(rk))
        return self._ok("hba_rdm_spearman")

    # ---------------------------------------------------------------- helpers
    def hba_add_rows(self, dst, ld_dst, dst_row_step, src, ld_src, rows, cols, stream):
        _require(_addr(dst) and _addr(src) and rows > 0 and cols > 0, "bad arguments")
        dst_row_step = max(1, dst_row_step)
        d = flat(dst, ((rows - 1) * dst_row_step) * ld_dst + cols, torch.float32).as_strided(
            (rows, cols), (ld_dst * dst_row_step, 1))
        d.add_(mat(src, rows, cols, ld_src, torch.float32))
        return self._ok("hba_add_rows")

    def hba_nonfinite_flag(self, x, n, flag, stream):
        if not bool(torch.isfinite(flat(x, n, torch.float32)).all()):
            flat(flag, 1, torch.int32)[0] = 1
        return self._ok("hba_nonfinite_flag")


@contextlib.contextmanager
def emulated_device():
    """Runs the product's host side on CPU tensors: libhba's entry points are served by `RefLib`, the `is_cuda` /
    current-device / stream plumbing answers as if the CPU were the one CUDA device, CUDA-graph capture and the
    side stream are switched off (HBA_STEP_GRAPH=0, HBA_TEXT_STREAM=0).  Test processes only."""
    import hba._lib as lib_mod
    import hba.ops as ops
    saved = {"lib": lib_mod._lib, "p": ops._p, "stream": ops._stream, "is_cuda": torch.Tensor.is_cuda,
             "cur": torch.cuda.current_device, "dev": torch.cuda.device, "sync": torch.cuda.synchronize,
             "env": {k: os.environ.get(k) for k in ("HBA_STEP_GRAPH", "HBA_TEXT_STREAM")}}
    ref = RefLib()
    lib_mod._lib = ref
    ops._p = lambda t: None if t is None else t.data_ptr()
    ops._stream = lambda: None
    torch.Tensor.is_cuda = property(lambda self: True)
    torch.cuda.current_device = lambda: None
    torch.cuda.device = lambda *_a, **_k: contextlib.nullcontext()
    torch.cuda.synchronize = lambda *_a, **_k: None
    os.environ.update(HBA_STEP_GRAPH="0", HBA_TEXT_STREAM="0")
    try:
        yield ref
    finally:
        lib_mod._lib, ops._p, ops._stream = saved["lib"], saved["p"], saved["stream"]
        torch.Tensor.is_cuda = saved["is_cuda"]
        torch.cuda.current_device, torch.cuda.device, torch.cuda.synchronize = saved["cur"], saved["dev"], saved["sync"]
        for k, v in saved["env"].items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
