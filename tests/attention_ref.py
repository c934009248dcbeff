"""fp64 reference of the libhba attention kernels, and the branch map of their launchers.

`reference()` is softmax attention as F.multi_head_attention_forward reaches it (scaled by 1/8,
optional CLIP causal mask) on the exact values handed to a kernel, in fp64 on whatever device they are
on.  `tc_fwd_branches()` / `tc_bwd_branches()` restate how the tcgen05 launchers (attention_tc.cu,
attention_bwd_tc.cu) split a sequence length T into tiles, left-over rows, tensor-core keys and TMA
boxes; `simt_bwd_fits()` restates the shared-memory size of the CUDA-core backward (vit_extra.cu).
`spiked_qkv()` builds inputs that concentrate chosen rows' softmax mass on chosen keys, so that a
kernel branch that mishandles one key or one query row shows an O(1) error instead of an O(1/T) one.
"""
from __future__ import annotations

import math

import torch

HD = 64
LOG2E = 1.4426950408889634
SMEM_LIMIT = 227 * 1024      # dynamic shared memory of one CTA on sm_100
SIMT_MAX_T = 288             # CUDA-core kernels: 9 key chunks of 32 per lane
TC_FWD_MAX_T = 257
TC_BWD_MAX_T = 256


def _heads(x, B, T, H):
    """[B*T, H*64] (any row stride) -> [B, H, T, 64] fp64."""
    return x.double().reshape(B, T, H, HD).permute(0, 2, 1, 3)


def _rows(x, B, T, H):
    """[B, H, T, 64] -> [B*T, H*64]."""
    return x.permute(0, 2, 1, 3).reshape(B * T, H * HD)


def reference(qkv, B, T, H, causal=False, d_out=None, o_for_d=None):
    """Softmax attention of qkv [B*T, 3*H*64] in fp64.

    Returns a dict with o [B*T, H*64], lse [B, H, T] (log2 of the softmax denominator of s / 8, the
    statistic hba_attention_fwd_lse writes) and, when d_out [B*T, H*64] is given, dqkv [B*T, 3*H*64]
    by autograd.  `o_for_d` (the forward output handed to a backward kernel) replaces the exact O in
    D_i = dO_i . O_i of the FlashAttention-2 backward dS = P o (dP - D): the gradient of the operation
    that kernel computes from the values it is given.
    """
    d = H * HD
    x = qkv[:, :3 * d].double().detach().clone().requires_grad_(d_out is not None)
    q, k, v = (_heads(x[:, i * d:(i + 1) * d], B, T, H) for i in range(3))
    s = (q @ k.transpose(-1, -2)) / 8.0
    if causal:
        s = s + torch.full((T, T), float("-inf"), dtype=torch.float64, device=s.device).triu_(1)
    p = s.softmax(-1)
    o = p @ v
    res = {"o": _rows(o, B, T, H).detach(), "lse": (torch.logsumexp(s, -1) * LOG2E).detach()}
    if d_out is None:
        return res
    do = _heads(d_out, B, T, H)
    if o_for_d is None:
        o.backward(do)
        res["dqkv"] = x.grad.detach()
        return res
    # explicit backward with D taken from the given O (equal to autograd when o_for_d is exact)
    vv = v.detach()
    dv = p.transpose(-1, -2) @ do
    dp = do @ vv.transpose(-1, -2)
    dd = (do * _heads(o_for_d, B, T, H)).sum(-1, keepdim=True)
    ds = p * (dp - dd) / 8.0
    dq = ds @ k.detach()
    dk = ds.transpose(-1, -2) @ q.detach()
    res["dqkv"] = torch.cat([_rows(dq, B, T, H), _rows(dk, B, T, H), _rows(dv, B, T, H)], 1).detach()
    return res


def reference_row0(qkv, B, T, H, d_out=None):
    """Query row 0 of every sequence (first_row_only): o [B, H*64]; dqkv [B*T, 3*H*64] when d_out [B, H*64]
    is given (zero dq on rows > 0)."""
    d = H * HD
    x = qkv[:, :3 * d].double().detach().clone().requires_grad_(d_out is not None)
    q, k, v = (_heads(x[:, i * d:(i + 1) * d], B, T, H) for i in range(3))
    o = ((q[:, :, :1] @ k.transpose(-1, -2)) / 8.0).softmax(-1) @ v   # [B, H, 1, 64]
    o = o.reshape(B, H * HD)
    res = {"o": o.detach()}
    if d_out is not None:
        o.backward(d_out.double())
        res["dqkv"] = x.grad.detach()
    return res


# ---------------------------------------------------------------------------------------- branch map
def tc_fwd_branches(T):
    """attention_tc_launch's split of T; `ok` is False where the launcher returns HBA_ERR_ARG."""
    rem = T % 128
    if T > 128 and 0 < rem <= 8:
        n_tiles, n_left = T // 128, rem
    else:
        n_tiles, n_left = (T + 127) // 128, 0
    kv_rows = (T + 15) // 16 * 16
    NK = min(kv_rows, 256)
    n_extra = max(T - NK, 0)
    return {"n_tiles": n_tiles, "n_left": n_left, "kv_rows": kv_rows, "NK": NK, "n_extra": n_extra,
            "tail_boxes": (kv_rows % 128) // 16, "nk_mod32": NK % 32 == 0,
            "ok": n_tiles <= 2 and n_extra <= 1 and kv_rows <= 272}


def tc_bwd_branches(T):
    """attention_bwd_tc_launch's split of T: rows = T rounded up to 16, one or two 128-row tiles of
    keys and of queries, the second (rows1 rows) partial unless T is 256."""
    rows = (T + 15) // 16 * 16
    rows0 = min(rows, 128)
    return {"rows": rows, "n_tiles": 2 if rows > 128 else 1, "rows0": rows0, "rows1": rows - rows0,
            "tail_rows": rows - T, "ok": T <= TC_BWD_MAX_T}


def simt_bwd_fits(T, dtype):
    """Whether hba_attention_bwd's shared memory (Q, K, V, dO tiles, three row statistics and two
    per-warp score buffers) fits one CTA: fp32 (qkv_dtype f32) up to T = 203, bf16 up to 288."""
    pitch = 65 if dtype == torch.float32 else 33
    smem = 4 * 4 * T * pitch + 4 * 3 * T + 4 * 8 * 2 * SIMT_MAX_T
    return T <= SIMT_MAX_T and smem <= SMEM_LIMIT


# ---------------------------------------------------------------------------------------- inputs
def spiked_qkv(B, T, H, pairs, *, seed=0, dtype=torch.bfloat16, device="cpu"):
    """qkv [B*T, 3*H*64] of N(0, 0.5^2) entries in which, in every sequence and head, query row r of each
    (r, j) in `pairs` carries more than 90 % of its softmax mass on key j: k_j = 8 u and q_r = 10 u for a
    random unit vector u, so s_rj / 8 = 10 while the other scores of row r have a standard deviation of
    about 0.6.  Each row and each key may appear in one pair only."""
    rows = [r for r, _ in pairs]
    keys = [j for _, j in pairs]
    assert len(set(rows)) == len(rows) and len(set(keys)) == len(keys), pairs
    assert all(0 <= r < T and 0 <= j < T for r, j in pairs), (T, pairs)
    g = torch.Generator().manual_seed(seed)
    d = H * HD
    x = torch.randn(B, T, 3, H, HD, generator=g, dtype=torch.float64) * 0.5
    for r, j in pairs:
        u = torch.randn(B, H, HD, generator=g, dtype=torch.float64)
        u = u / u.norm(dim=-1, keepdim=True)
        x[:, j, 1] = 8.0 * u
        x[:, r, 0] = 10.0 * u
    return x.reshape(B * T, 3 * d).to(dtype).to(device)


def spike_pairs(T, causal, keys=(0, 15, 16, 127, 128, 255, 256), rows=(0, 127, 128, 255, 256)):
    """(query row, key) pairs for a length-T sweep point: the keys 0, 15, 16, 127, 128, NK-1, 256 and T-1
    and the query rows 0, 127, 128, 255, 256 and T-1 that exist at T.  Causal: each index is paired
    with itself (a key is visible to its own row).  Otherwise the sorted indices are paired with the
    same list reversed, so that e.g. at T = 257 row 0 (tensor-core tile 0) puts its mass on key 256
    (the fp32 extra key) and row 256 (the CUDA-core left-over row) on key 0."""
    nk = tc_fwd_branches(T)["NK"] if T <= TC_FWD_MAX_T else min((T + 15) // 16 * 16, 256)
    idx = sorted({i for i in (*keys, *rows, nk - 1, T - 1) if 0 <= i < T})
    if causal:
        return [(i, i) for i in idx]
    return list(zip(idx, reversed(idx)))


def softmax_mass(qkv, B, T, H, causal=False):
    """P [B, H, T, T] in fp64 (the softmax the spikes are designed for)."""
    d = H * HD
    q, k = (_heads(qkv[:, i * d:(i + 1) * d], B, T, H) for i in range(2))
    s = (q @ k.transpose(-1, -2)) / 8.0
    if causal:
        s = s + torch.full((T, T), float("-inf"), dtype=torch.float64, device=s.device).triu_(1)
    return s.softmax(-1)


# ---------------------------------------------------------------------------------------- errors
def row_err(got, want, width=HD):
    """Worst per-row error: rows are consecutive `width`-element segments (one head of one token);
    for each, max |got - want| over max |want_row|, that maximum clamped to at least 1e-3 of the largest
    |want| in the tensor (rows whose reference is exactly zero must then be zero to within 1e-3 * tol)."""
    g = got.detach().double().to(want.device).reshape(-1, width)
    w = want.detach().double().reshape(-1, width)
    if g.shape != w.shape:
        raise ValueError((got.shape, want.shape))
    scale = w.abs().amax(1).clamp_min(max(float(w.abs().max()) * 1e-3, 1e-30))
    e = (g - w).abs().amax(1) / scale
    if not bool(torch.isfinite(g).all()):
        return math.inf
    return float(e.max())
