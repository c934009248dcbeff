"""Torch-tensor front ends of the libhba C-ABI (device memory + stream plumbing only).

Every function takes CUDA tensors, passes raw pointers / leading dimensions / the current stream to
the C-ABI and raises ``RuntimeError`` on failure.  Nothing here computes on the host.
"""
from __future__ import annotations

import ctypes as C
import functools
import itertools

import torch

from . import _lib
from ._lib import (HBA_ACT_GELU_ERF, HBA_ACT_GELU_ERF_GRAD, HBA_ACT_NONE, HBA_ACT_QUICKGELU,
                   HBA_ACT_QUICKGELU_GRAD, HBA_DT_BF16, HBA_DT_F32, GemmParams)
from ._lib import check as _check

# Our own count of kernels launched through the C-ABI (bench.py reports it as `gpu_launches`).
COUNTERS = {"launches": 0, "calls": 0}
_KERNELS_PER_CALL = {"hba_dora_merge_bwd": 2, "hba_pearson_f64": 3, "hba_softmax_ce_fwd_bwd": 2}
# When set to a list, every GEMM launch is bracketed by CUDA events on the launching stream and
# (M, N, K, nsplit, start_event, end_event) is appended (bench.py's live roofline measurement).
GEMM_PROFILE = None
# Upper bound on the CTAs of every GEMM launched without an explicit `max_ctas` (0 = all SMs).  The data-parallel
# ViT trainer lowers it during a multi-rank backward pass so that NCCL's all-reduce CTAs find free SMs beside the
# persistent GEMM kernels instead of queueing behind them (HBA_DP_GEMM_CTAS).
GEMM_MAX_CTAS = 0


class EventProfile:
    """Context manager: every C-ABI launch made through this module is bracketed by CUDA events on the
    launching stream; `.records` holds (entry point, start, end).  Used by bench.py for the kernel-time
    shares of a step (a measurement aid - the events add host work, never use it in a timed region)."""

    def __init__(self):
        self.records = []

    def __enter__(self):
        global _lib
        real, records = _lib, self.records

        class _Lib:
            def __getattr__(self, name):
                fn = getattr(real.load(), name)
                if not name.startswith("hba_") or name == "hba_last_error" or name.endswith("_workspace_bytes"):
                    return fn

                def bracketed(*args):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    rc = fn(*args)
                    e1.record()
                    records.append((name, e0, e1))
                    return rc
                return bracketed

        class _Shim:
            def __getattr__(self, name):
                return getattr(real, name)

            @staticmethod
            def load():
                return _Lib()

        self._real = real
        _lib = _Shim()
        return self

    def __exit__(self, *exc):
        global _lib
        _lib = self._real
        return False

    def totals_ms(self):
        out = {}
        for name, e0, e1 in self.records:
            out[name] = out.get(name, 0.0) + e0.elapsed_time(e1)
        return out


def check(rc, what, kernels=None):
    _check(rc, what)
    COUNTERS["calls"] += 1
    COUNTERS["launches"] += kernels if kernels is not None else _KERNELS_PER_CALL.get(what, 1)

__all__ = ["gemm", "split_bf16", "layernorm_fwd", "layernorm_bwd", "im2col_patches",
           "assemble_tokens_ln", "embed_tokens", "gather_rows", "attention_fwd",
           "attention_bwd_row0", "dora_merge_fwd", "dora_merge_bwd", "cos_head_fwd", "cos_head_bwd", "cos_mse_fwd", "cos_mse_bwd",
           "adamw_multi", "sgd_multi", "rdm_f64", "rank_avg_f64", "pearson_f64", "softmax_ce",
           "add_rows", "nonfinite_flag", "Operand"]


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    if t is None:
        return None
    assert t.is_cuda, "libhba operates on CUDA tensors only (no CPU fallback)"
    return C.c_void_p(t.data_ptr())


def _dt(t):
    if t.dtype == torch.float32:
        return HBA_DT_F32
    if t.dtype == torch.bfloat16:
        return HBA_DT_BF16
    raise TypeError(f"unsupported dtype {t.dtype}")


class Operand:
    """A bf16 GEMM operand [rows, K] with an optional lo part (fp32 mode): ``buf`` is
    [rows, ld] bf16 with hi at columns [0, K) and, when ``lo_off > 0``, lo at [lo_off, lo_off+K)."""
    __slots__ = ("buf", "rows", "K", "lo_off")

    def __init__(self, buf, rows, K, lo_off):
        self.buf, self.rows, self.K, self.lo_off = buf, rows, K, lo_off

    @property
    def ld(self):
        return self.buf.stride(0)

    @staticmethod
    def empty(rows, K, split, device, zero=False):
        width = 2 * K if split else K
        f = torch.zeros if zero else torch.empty
        return Operand(f(rows, width, dtype=torch.bfloat16, device=device), rows, K, K if split else 0)

    def narrow_rows(self, start, n):
        return Operand(self.buf.narrow(0, start, n), n, self.K, self.lo_off)


def auto_k_slices(M, N, K, workers=74, max_slices=16, min_kblocks=8):
    """Split-K factor for a weight-gradient GEMM (or, with min_kblocks=4, a skinny row GEMM): minimises
    rounds-of-work-items / slices (the time of the persistent kernel in units of one full-K tile) plus a small
    per-slice epilogue / reduction cost."""
    tiles = -(-M // 256) * -(-N // (256 if N >= 256 else 128))
    kblocks = -(-K // 64)
    best, best_cost = 1, None
    for s in range(1, max_slices + 1):
        if s > 1 and (kblocks // s < min_kblocks or N % 4):
            break
        cost = -(-tiles * s // workers) / s + 0.02 * (s - 1)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = s, cost
    return best


def gemm(a: Operand, b: Operand, M=None, *, bias=None, residual=None, act=HBA_ACT_NONE, aux=None,
         pre_out=None, out_f32=None, out: Operand = None, transpose_out=False, alpha=1.0,
         max_ctas=0, a_mn=False, b_mn=False, K=None, k_slices=1, k_workspace=None, colsum_partial=None):
    """C[M,N] = epilogue(A . B^T) on the tcgen05 tensor pipe (hba_gemm_bf16).
    a_mn / b_mn: the operand is stored MN-major, i.e. as [K rows, M resp. N columns] (its Operand
    then has rows = K and K = M resp. N)."""
    if a_mn:
        Ka, M = a.rows, (a.K if M is None else M)
    else:
        Ka, M = a.K, (a.rows if M is None else M)
    Kb, N = (b.rows, b.K) if b_mn else (b.K, b.rows)
    K = min(Ka, Kb) if K is None else K
    assert K <= Ka and K <= Kb, (K, Ka, Kb)
    if K % 64 and a.lo_off > 0 and b.lo_off > 0:
        # ragged K in fp32 mode: a K-major operand must be zero padded up to its lo part
        assert a_mn or a.lo_off >= (K + 63) // 64 * 64, "A needs zero padding up to a multiple of 64"
        assert b_mn or b.lo_off >= (K + 63) // 64 * 64, "B needs zero padding up to a multiple of 64"
    split = a.lo_off > 0 and b.lo_off > 0
    p = GemmParams()
    p.A, p.B = a.buf.data_ptr(), b.buf.data_ptr()
    p.M, p.N, p.K = M, N, K
    p.lda, p.ldb = a.ld, b.ld
    p.nsplit = 3 if split else 1
    p.a_lo_off, p.b_lo_off = (a.lo_off, b.lo_off) if split else (0, 0)
    p.alpha = alpha
    p.bias = bias.data_ptr() if bias is not None else None
    if residual is not None:
        p.residual, p.ldr = residual.data_ptr(), residual.stride(0)
    p.act = act
    if aux is not None:
        p.aux, p.ld_aux, p.aux_dtype = aux.data_ptr(), aux.stride(0), _dt(aux)
    if pre_out is not None:
        p.pre_out, p.ld_pre, p.pre_dtype = pre_out.data_ptr(), pre_out.stride(0), _dt(pre_out)
    if out_f32 is not None:
        p.out_f32, p.ld_f32 = out_f32.data_ptr(), out_f32.stride(0)
    if out is not None:
        p.out_bf16, p.ld_bf16, p.out_lo_off = out.buf.data_ptr(), out.ld, out.lo_off
    p.transpose_out = 1 if transpose_out else 0
    p.max_ctas = max_ctas or GEMM_MAX_CTAS
    p.a_mn_major, p.b_mn_major = (1 if a_mn else 0), (1 if b_mn else 0)
    launches = 1
    if colsum_partial is not None:
        assert colsum_partial.dtype == torch.float32 and colsum_partial.numel() >= (M + 31) // 32 * N
        p.colsum_partial = colsum_partial.data_ptr()
    if k_slices == "auto":
        k_slices = auto_k_slices(M, N, K)
    if k_slices > 1:
        assert k_workspace is not None and k_workspace.dtype == torch.float32
        assert k_workspace.numel() >= k_slices * M * N, "k_workspace too small"
        p.k_slices, p.k_workspace = k_slices, k_workspace.data_ptr()
        launches = 2
    if GEMM_PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        check(_lib.load().hba_gemm_bf16(C.byref(p), _stream()), "hba_gemm_bf16", launches)
        e1.record()
        GEMM_PROFILE.append((M, N, K, p.nsplit, e0, e1))
        return
    check(_lib.load().hba_gemm_bf16(C.byref(p), _stream()), "hba_gemm_bf16", launches)


def split_bf16(x, out: Operand, transpose=False):
    """fp32 [rows, cols] -> bf16 hi(/lo) operand; ``transpose`` writes out[c, r]."""
    rows, cols = x.shape
    check(_lib.load().hba_split_bf16(_p(x), rows, cols, x.stride(0), _p(out.buf), out.ld, out.lo_off,
                                     1 if transpose else 0, _stream()), "hba_split_bf16")
    return out


def layernorm_fwd(x, rows, cols, gamma, beta, eps, *, row_step=1, y_f32=None, y: Operand = None):
    check(_lib.load().hba_layernorm_fwd(
        _p(x), rows, cols, x.stride(0), row_step, _p(gamma), _p(beta), eps,
        _p(y_f32), y_f32.stride(0) if y_f32 is not None else 0,
        _p(y.buf) if y is not None else None, y.ld if y is not None else 0,
        y.lo_off if y is not None else 0, _stream()), "hba_layernorm_fwd")


def layernorm_bwd(dy, x, rows, cols, gamma, eps, dx, *, row_step=1, accumulate=False):
    check(_lib.load().hba_layernorm_bwd(_p(dy), dy.stride(0), _p(x), rows, cols, x.stride(0), row_step,
                                        _p(gamma), eps, _p(dx), dx.stride(0), 1 if accumulate else 0,
                                        _stream()), "hba_layernorm_bwd")


def im2col_patches(image, P, out: Operand):
    B, Cc, H, W = image.shape
    assert Cc == 3 and image.is_contiguous() and image.dtype == torch.float32
    check(_lib.load().hba_im2col_patches(_p(image), B, H, W, P, _p(out.buf), out.ld, out.lo_off,
                                         _stream()), "hba_im2col_patches")


def assemble_tokens_ln(conv, B, n_patches, width, cls, pos, gamma, beta, eps, x_out):
    check(_lib.load().hba_assemble_tokens_ln(_p(conv), B, n_patches, width, _p(cls), _p(pos), _p(gamma),
                                             _p(beta), eps, _p(x_out), _stream()),
          "hba_assemble_tokens_ln")


def embed_tokens(tokens, table, pos, x_out):
    S, T = tokens.shape
    assert tokens.dtype == torch.int64 and tokens.is_contiguous()
    check(_lib.load().hba_embed_tokens(_p(tokens), S, T, table.shape[1], _p(table), _p(pos), _p(x_out),
                                       _stream()), "hba_embed_tokens")


def gather_rows(src, idx, cols, out):
    check(_lib.load().hba_gather_rows(_p(src), src.stride(0), _p(idx), idx.numel(), cols, _p(out),
                                      out.stride(0), _stream()), "hba_gather_rows")


def attention_fwd(qkv, B, T, H, *, causal=False, first_row_only=False, out: Operand = None,
                  out_f32=None):
    check(_lib.load().hba_attention_fwd(
        _p(qkv), _dt(qkv), qkv.stride(0), B, T, H, 1 if causal else 0, 1 if first_row_only else 0,
        _p(out.buf) if out is not None else None, out.ld if out is not None else 0,
        out.lo_off if out is not None else 0, _p(out_f32),
        out_f32.stride(0) if out_f32 is not None else 0, _stream()), "hba_attention_fwd")


def attention_bwd_row0(qkv, B, T, H, d_out, d_qkv):
    check(_lib.load().hba_attention_bwd_row0(_p(qkv), _dt(qkv), qkv.stride(0), B, T, H, _p(d_out),
                                             d_out.stride(0), _p(d_qkv), d_qkv.stride(0), _stream()),
          "hba_attention_bwd_row0")


def dora_merge_fwd(D, A, Bm, m, scale, eps, *, w_t_f32=None, w: Operand = None, wt: Operand = None,
                   norm_out=None):
    in_f, out_f = D.shape
    r = A.shape[0]
    check(_lib.load().hba_dora_merge_fwd(
        _p(D), _p(A), _p(Bm), _p(m), in_f, out_f, r, scale, eps, _p(w_t_f32),
        _p(w.buf) if w is not None else None, w.ld if w is not None else 0,
        w.lo_off if w is not None else 0,
        _p(wt.buf) if wt is not None else None, wt.ld if wt is not None else 0,
        wt.lo_off if wt is not None else 0, _p(norm_out), _stream()), "hba_dora_merge_fwd")


def dora_merge_bwd(G, D, A, Bm, m, scale, eps, dm, dA, dB, workspace):
    in_f, out_f = D.shape
    check(_lib.load().hba_dora_merge_bwd(_p(G), G.stride(0), _p(D), _p(A), _p(Bm), _p(m), in_f, out_f,
                                         A.shape[0], scale, eps, _p(dm), _p(dA), _p(dB), _p(workspace),
                                         _stream()), "hba_dora_merge_bwd")


def cos_head_fwd(img, txt, logit_scale, pred, target=None, loss=None):
    B, E = img.shape
    check(_lib.load().hba_cos_head_fwd(_p(img), _p(txt), B, txt.shape[0], E, _p(logit_scale), _p(pred),
                                       _p(target), _p(loss), _stream()), "hba_cos_head_fwd",
          2 if loss is not None else 1)


def cos_head_bwd(img, txt, logit_scale, d_img, d_txt, *, d_pred=None, pred=None, target=None):
    B, E = img.shape
    check(_lib.load().hba_cos_head_bwd(_p(img), _p(txt), B, txt.shape[0], E, _p(logit_scale),
                                       _p(d_pred), _p(pred), _p(target), _p(d_img), _p(d_txt),
                                       _stream()), "hba_cos_head_bwd")


def cos_mse_fwd(img, txt, logit_scale, pred, *, B, groups=1, target=None, target_group_stride=0, loss=None,
                bad_step=None, bad_total=None, total=None, workspace=None):
    """Cosine logits (+ fused nn.MSELoss, non-finite flag and running loss sum) in one launch; `groups`
    independent problems laid out contiguously: img [groups*B, E], txt [groups*C, E], pred [groups*B, C]."""
    E = img.shape[-1]
    C_ = txt.shape[0] // groups
    assert img.shape[0] == groups * B and txt.shape[0] == groups * C_ and pred.numel() == groups * B * C_
    if target is not None:
        assert target.dtype == torch.float32 and target.is_contiguous()
        assert workspace is not None and workspace.numel() >= groups * (B + 1)
    check(_lib.load().hba_cos_mse_fwd(_p(img), _p(txt), B, C_, E, groups, _p(logit_scale), _p(pred), _p(target),
                                      target_group_stride, _p(loss), _p(bad_step), _p(bad_total), _p(total),
                                      _p(workspace), _stream()), "hba_cos_mse_fwd")


def cos_mse_bwd(img, txt, logit_scale, pred, target, d_img, d_txt, *, B, groups=1, target_group_stride=0,
                d_loss=None):
    E = img.shape[-1]
    C_ = txt.shape[0] // groups
    check(_lib.load().hba_cos_mse_bwd(_p(img), _p(txt), B, C_, E, groups, _p(logit_scale), _p(pred), _p(target),
                                      target_group_stride, _p(d_loss), _p(d_img), _p(d_txt), _stream()),
          "hba_cos_mse_bwd")


def adamw_multi(ptr_table, sizes, n, total, lr, beta1, beta2, eps, weight_decay, step, skip_flag=None,
                step_dev=None):
    """step: host step count (>= 1), or 0 with step_dev = device int32 holding the count."""
    check(_lib.load().hba_adamw_multi(_p(ptr_table), _p(sizes), n, total, lr, beta1, beta2, eps,
                                      weight_decay, step, _p(step_dev), _p(skip_flag), _stream()),
          "hba_adamw_multi")


def sgd_multi(ptr_table, sizes, n, total, lr, momentum, weight_decay, first_step, skip_flag=None):
    check(_lib.load().hba_sgd_multi(_p(ptr_table), _p(sizes), n, total, lr, momentum, weight_decay,
                                    1 if first_step else 0, _p(skip_flag), _stream()), "hba_sgd_multi")


def sgd_staged(ptr_table, prefix4, n, total4, lr, momentum, weight_decay, first_step, skip_flag=None):
    check(_lib.load().hba_sgd_staged(_p(ptr_table), _p(prefix4), n, total4, lr, momentum, weight_decay,
                                     1 if first_step else 0, _p(skip_flag), _stream()), "hba_sgd_staged")


def rdm_f64(E, rdm=None, tri=None):
    N, Dm = E.shape
    assert E.dtype == torch.float32 and E.is_contiguous()
    check(_lib.load().hba_rdm_f64(_p(E), N, Dm, _p(rdm), _p(tri), _stream()), "hba_rdm_f64")


def rank_workspace_bytes(n):
    return int(_lib.load().hba_rank_workspace_bytes(n))


def rank_avg_f64(x, ranks, workspace=None):
    n = x.numel()
    assert x.dtype == torch.float64 and ranks.dtype == torch.float64
    need = rank_workspace_bytes(n)
    if workspace is None:
        workspace = torch.empty(need, dtype=torch.uint8, device=x.device)
    check(_lib.load().hba_rank_avg_f64(_p(x), n, _p(ranks), _p(workspace), workspace.numel(), _stream()),
          "hba_rank_avg_f64", 1 if n <= 2048 else 10)


def pearson_f64(a, b, rho_out, workspace):
    check(_lib.load().hba_pearson_f64(_p(a), _p(b), a.numel(), _p(rho_out), _p(workspace), _stream()),
          "hba_pearson_f64")


def rdm_spearman(E, ref_ranks, rho_out, workspace, rdm=None, ranks=None):
    """RSA at scale, one checkpoint: E [N, Dm] fp32 -> rho (device double) against ref_ranks [N(N-1)/2] f64."""
    N, Dm = E.shape
    assert E.dtype == torch.float32 and E.is_contiguous() and ref_ranks.dtype == torch.float64
    assert ref_ranks.numel() == N * (N - 1) // 2
    check(_lib.load().hba_rdm_spearman(_p(E), N, Dm, _p(ref_ranks), _p(rdm), _p(ranks), _p(rho_out), _p(workspace),
                                       workspace.numel(), _stream()), "hba_rdm_spearman", 11)


def rank_order_f64(x, order, ranks, workspace):
    """ranks as rank_avg_f64, and order [n] int32 (uint32 bits): the stable sorted order of x."""
    n = x.numel()
    assert x.dtype == torch.float64 and ranks.dtype == torch.float64 and order.dtype == torch.int32
    assert x.is_contiguous() and order.numel() == n and ranks.numel() == n
    check(_lib.load().hba_rank_order_f64(_p(x), n, _p(order), _p(ranks), _p(workspace), workspace.numel(), _stream()),
          "hba_rank_order_f64", 1 if n <= 2048 else 11)


def rsa_perm_workspace_bytes(N, n_perm):
    return int(_lib.load().hba_rsa_perm_workspace_bytes(N, n_perm))


def rsa_perm_null(ref_ranks, model_ranks, perms, rho_out, workspace):
    """Mantel null: rho_out[p] = Spearman rho of the reference against the model relabelled by perms[p]
    (perms [n_perm, N] int32, every row a permutation - the caller checks that)."""
    n_perm, N = perms.shape
    P = N * (N - 1) // 2
    assert ref_ranks.dtype == model_ranks.dtype == rho_out.dtype == torch.float64 and perms.dtype == torch.int32
    assert ref_ranks.numel() == model_ranks.numel() == P and rho_out.numel() >= n_perm and perms.is_contiguous()
    check(_lib.load().hba_rsa_perm_null(_p(ref_ranks), _p(model_ranks), N, _p(perms), n_perm, _p(rho_out),
                                        _p(workspace), workspace.numel(), _stream()), "hba_rsa_perm_null", 3)


def rsa_boot_workspace_bytes(N, n_boot):
    return int(_lib.load().hba_rsa_boot_workspace_bytes(N, n_boot))


def rsa_bootstrap(ref_tri, ref_order, tri_a, order_a, counts, rho_a, workspace, tri_b=None, order_b=None, rho_b=None):
    """Stimulus bootstrap: rho_a[b] (and rho_b[b]) = Spearman rho of the reference against model a (b) over the
    pairs of the resample with counts[b] (counts [n_boot, N] int32, each row summing to N)."""
    n_boot, N = counts.shape
    P = N * (N - 1) // 2
    assert counts.dtype == torch.int32 and counts.is_contiguous() and rho_a.numel() >= n_boot
    for t in (ref_tri, tri_a, tri_b):
        assert t is None or (t.dtype == torch.float64 and t.numel() == P)
    for t in (ref_order, order_a, order_b):
        assert t is None or (t.dtype == torch.int32 and t.numel() == P)
    kernels = 2 + 6 * (3 if tri_b is not None else 2)
    check(_lib.load().hba_rsa_bootstrap(_p(ref_tri), _p(ref_order), _p(tri_a), _p(order_a), _p(tri_b), _p(order_b), N,
                                        _p(counts), n_boot, _p(rho_a), _p(rho_b), _p(workspace), workspace.numel(),
                                        _stream()), "hba_rsa_bootstrap", kernels)


def kendall_workspace_bytes(n):
    return int(_lib.load().hba_kendall_workspace_bytes(n))


def kendall_kernels(n):
    """Kernels one hba_kendall_tau_f64 call launches: one CTA up to n = 2048; else keys, the radix sort (histogram +
    8 digit passes), y-ranks, tiles of 4096, one merge level per doubling of the run width up to n, final."""
    if n <= 2048:
        return 1
    levels, width = 0, 4096
    while width < n:
        levels, width = levels + 1, 2 * width
    return 13 + levels


def kendall_tau_f64(x, y, y_order, counts, tau, workspace):
    """Kendall's tau of x against y [n] f64 from exact pair counts: counts [4] int64 = (S, n1, n2, n3), tau [2] f64 =
    (tau_a, tau_b); y_order [n] int32 (uint32 bits) is y's stable sorted order (rank_order_f64)."""
    n = x.numel()
    assert x.dtype == y.dtype == tau.dtype == torch.float64 and y_order.dtype == torch.int32
    assert counts.dtype == torch.int64 and counts.numel() >= 4 and tau.numel() >= 2
    assert x.is_contiguous() and y.is_contiguous() and y_order.is_contiguous()
    assert y.numel() == n and y_order.numel() == n
    check(_lib.load().hba_kendall_tau_f64(_p(x), _p(y), _p(y_order), n, _p(counts), _p(tau), _p(workspace),
                                          workspace.numel() if workspace is not None else 0, _stream()),
          "hba_kendall_tau_f64", kendall_kernels(n))


def softmax_ce(logits, labels, loss, d_logits, correct, workspace):
    B, Cc = logits.shape
    check(_lib.load().hba_softmax_ce_fwd_bwd(_p(logits), logits.stride(0), _p(labels), B, Cc, _p(loss),
                                             _p(d_logits),
                                             d_logits.stride(0) if d_logits is not None else 0,
                                             _p(correct), _p(workspace), _stream()),
          "hba_softmax_ce_fwd_bwd")


def colsum(x, out, workspace, accumulate=False):
    rows, cols = x.shape
    check(_lib.load().hba_colsum(_p(x), _dt(x), rows, cols, x.stride(0), _p(out), 1 if accumulate else 0,
                                 _p(workspace), _stream()), "hba_colsum", 2)


def layernorm_param_grad(dy, x, rows, cols, eps, dgamma_dbeta, workspace, *, row_step=1, accumulate=False):
    check(_lib.load().hba_layernorm_param_grad(_p(dy), dy.stride(0), _p(x), rows, cols, x.stride(0),
                                               row_step, eps, _p(dgamma_dbeta), 1 if accumulate else 0,
                                               _p(workspace), _stream()), "hba_layernorm_param_grad", 3)


def attention_bwd(qkv, B, T, H, d_out, d_qkv, causal=False):
    check(_lib.load().hba_attention_bwd(_p(qkv), _dt(qkv), qkv.stride(0), B, T, H, 1 if causal else 0,
                                        _p(d_out), _dt(d_out), d_out.stride(0), _p(d_qkv), _dt(d_qkv),
                                        d_qkv.stride(0), _stream()), "hba_attention_bwd")


def layernorm_bwd_fused(dy, x, rows, cols, gamma, eps, dx, dgamma_dbeta, workspace, *, accumulate=False,
                        dx_op: Operand = None, dx_colsum=None, accumulate_params=False):
    """One pass: dx (+)= LN backward, bf16 operand copy of dx, dgamma|dbeta, column sums of dx."""
    assert workspace.numel() >= 2 * 148 * 3 * cols
    check(_lib.load().hba_layernorm_bwd_fused(
        _p(dy), dy.stride(0), _p(x), rows, cols, x.stride(0), _p(gamma), eps, _p(dx), dx.stride(0),
        1 if accumulate else 0, _p(dx_op.buf) if dx_op is not None else None,
        dx_op.ld if dx_op is not None else 0, dx_op.lo_off if dx_op is not None else 0, _p(dgamma_dbeta),
        1 if accumulate_params else 0, _p(dx_colsum), _p(workspace), _stream()), "hba_layernorm_bwd_fused", 2)


def attention_fwd_lse(qkv, B, T, H, out, lse, causal=False):
    """bf16 tensor-core forward that also writes lse [B, H, T] (log2 domain) for attention_bwd_lse."""
    assert qkv.dtype == torch.bfloat16 and out.dtype == torch.bfloat16 and lse.dtype == torch.float32
    assert lse.is_contiguous() and lse.numel() >= B * H * T
    check(_lib.load().hba_attention_fwd_lse(_p(qkv), qkv.stride(0), B, T, H, 1 if causal else 0, _p(out),
                                            out.stride(0), _p(lse), _stream()), "hba_attention_fwd_lse")


def attention_bwd_lse(qkv, B, T, H, out, d_out, lse, d_qkv, causal=False):
    for t in (qkv, out, d_out, d_qkv):
        assert t.dtype == torch.bfloat16
    assert lse.dtype == torch.float32 and lse.is_contiguous()
    check(_lib.load().hba_attention_bwd_lse(_p(qkv), qkv.stride(0), B, T, H, 1 if causal else 0, _p(out),
                                            out.stride(0), _p(d_out), d_out.stride(0), _p(lse), _p(d_qkv),
                                            d_qkv.stride(0), _stream()), "hba_attention_bwd_lse")


def add_rows(dst, src, rows, cols, dst_row_step=1):
    check(_lib.load().hba_add_rows(_p(dst), dst.stride(0), dst_row_step, _p(src), src.stride(0), rows,
                                   cols, _stream()), "hba_add_rows")


def nonfinite_flag(x, flag):
    check(_lib.load().hba_nonfinite_flag(_p(x), x.numel(), _p(flag), _stream()), "hba_nonfinite_flag")


# ------------------------------------------------------------------------------------------------------
# Device guard.  The C-ABI launches on the calling thread's CURRENT device / the stream passed in, and
# `_stream()` is the current stream of the current device: a call whose tensors live on another GPU
# (config['cuda'] = 1 of the reference, NEW:1137-1144, while the process' current device is still 0) would
# launch in the wrong context.  Every front end therefore runs under `torch.cuda.device(<its tensors' device>)`
# and refuses operands that are spread over several devices.
def _device_guarded(fn):
    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for a in itertools.chain(args, kwargs.values()):
            t = a.buf if isinstance(a, Operand) else a
            if torch.is_tensor(t) and t.is_cuda:
                if dev is None:
                    dev = t.device
                elif t.device != dev:
                    raise RuntimeError(f"libhba {fn.__name__}: operands on different devices ({dev} and {t.device})")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


for _name in ("gemm", "split_bf16", "layernorm_fwd", "layernorm_bwd", "im2col_patches", "assemble_tokens_ln",
              "embed_tokens", "gather_rows", "attention_fwd", "attention_bwd_row0", "dora_merge_fwd", "dora_merge_bwd",
              "cos_head_fwd", "cos_head_bwd", "cos_mse_fwd", "cos_mse_bwd", "adamw_multi", "sgd_multi", "sgd_staged",
              "rdm_f64", "rank_avg_f64", "pearson_f64", "rdm_spearman", "rank_order_f64", "rsa_perm_null",
              "rsa_bootstrap", "kendall_tau_f64", "softmax_ce", "colsum", "layernorm_param_grad",
              "attention_bwd", "layernorm_bwd_fused", "attention_fwd_lse", "attention_bwd_lse", "add_rows",
              "nonfinite_flag"):
    globals()[_name] = _device_guarded(globals()[_name])
del _name
