"""The fp64 attention reference, the launchers' branch map and the spiked inputs that
tests/test_gpu_attention_shapes.py relies on, checked without a GPU."""
import itertools

import pytest
import torch

from attention_ref import (SIMT_MAX_T, TC_FWD_MAX_T, reference, reference_row0, simt_bwd_fits,
                           softmax_mass, spike_pairs, spiked_qkv, tc_bwd_branches, tc_fwd_branches)
from test_gpu_attention_shapes import SWEEP_T


def _sdpa(qkv, B, T, H, causal):
    d = H * 64
    q, k, v = (qkv[:, i * d:(i + 1) * d].reshape(B, T, H, 64).transpose(1, 2) for i in range(3))
    o = torch.nn.functional.scaled_dot_product_attention(q, k, v, is_causal=causal)
    return o.transpose(1, 2).reshape(B * T, d)


@pytest.mark.parametrize("B,T,H,causal", [(2, 1, 1, False), (2, 17, 2, True), (3, 77, 2, True),
                                          (2, 130, 1, False), (1, 257, 2, False)])
def test_reference_matches_sdpa_and_autograd(B, T, H, causal):
    g = torch.Generator().manual_seed(T)
    d = H * 64
    qkv = torch.randn(B * T, 3 * d, generator=g, dtype=torch.float64)
    do = torch.randn(B * T, d, generator=g, dtype=torch.float64)
    x = qkv.clone().requires_grad_(True)
    o = _sdpa(x, B, T, H, causal)
    o.backward(do)
    r = reference(qkv, B, T, H, causal, d_out=do)
    torch.testing.assert_close(r["o"], o.detach(), rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(r["dqkv"], x.grad, rtol=1e-10, atol=1e-10)
    # the explicit backward with D from the exact O is the same gradient
    r2 = reference(qkv, B, T, H, causal, d_out=do, o_for_d=r["o"])
    torch.testing.assert_close(r2["dqkv"], x.grad, rtol=1e-10, atol=1e-10)
    # lse: log2 of the softmax denominator of s / 8
    q, k = (qkv[:, i * d:(i + 1) * d].reshape(B, T, H, 64).transpose(1, 2) for i in range(2))
    s = q @ k.transpose(-1, -2) / 8
    if causal:
        s = s.masked_fill(torch.ones(T, T, dtype=torch.bool).triu(1), float("-inf"))
    torch.testing.assert_close(r["lse"], torch.logsumexp(s, -1) / torch.log(torch.tensor(2.0, dtype=torch.float64)))
    # first_row_only is row 0 of the full forward; its backward is autograd of that row
    if not causal:
        x0 = qkv.clone().requires_grad_(True)
        o0 = _sdpa(x0, B, T, H, False).view(B, T, d)[:, 0]
        do0 = do.view(B, T, d)[:, 0]
        o0.backward(do0)
        r0 = reference_row0(qkv, B, T, H, d_out=do0)
        torch.testing.assert_close(r0["o"], o0.detach(), rtol=1e-12, atol=1e-12)
        torch.testing.assert_close(r0["dqkv"], x0.grad, rtol=1e-10, atol=1e-10)


def test_reference_takes_strided_bf16_input():
    B, T, H = 2, 33, 2
    d = H * 64
    buf = torch.randn(B * T, 3 * d + 8, generator=torch.Generator().manual_seed(3)).to(torch.bfloat16)
    buf[:, 3 * d:] = float("nan")
    qkv = buf[:, :3 * d]
    want = _sdpa(qkv.double(), B, T, H, False)
    torch.testing.assert_close(reference(qkv, B, T, H)["o"], want, rtol=1e-12, atol=1e-12)


def _combos(Ts):
    out = set()
    for T in Ts:
        if T > TC_FWD_MAX_T:
            continue
        b = tc_fwd_branches(T)
        out.add((b["n_tiles"], b["n_left"], b["nk_mod32"], b["tail_boxes"] > 0, b["n_extra"]))
    return out


def test_branch_map_restates_the_launchers():
    assert tc_fwd_branches(257) == {"n_tiles": 2, "n_left": 1, "kv_rows": 272, "NK": 256, "n_extra": 1,
                                    "tail_boxes": 1, "nk_mod32": True, "ok": True}
    assert tc_fwd_branches(136)["n_left"] == 8 and tc_fwd_branches(137)["n_tiles"] == 2
    assert tc_fwd_branches(77)["NK"] == 80 and not tc_fwd_branches(77)["nk_mod32"]
    assert not tc_fwd_branches(258)["ok"] and tc_fwd_branches(256)["ok"]
    assert tc_bwd_branches(197) == {"rows": 208, "n_tiles": 2, "rows0": 128, "rows1": 80, "tail_rows": 11,
                                    "ok": True}
    assert not tc_bwd_branches(257)["ok"]
    # every T the tensor-core forward accepts is one of these combinations, and no other
    every = _combos(range(1, TC_FWD_MAX_T + 1))
    assert {c[0] for c in every} == {1, 2}
    assert {c[1] for c in every} == set(range(9))
    assert {c[2] for c in every} == {False, True} and {c[3] for c in every} == {False, True}
    assert {c[4] for c in every} == {0, 1}


def test_simt_bwd_shared_memory_limit():
    assert max(T for T in range(1, SIMT_MAX_T + 1) if simt_bwd_fits(T, torch.float32)) == 203
    assert all(simt_bwd_fits(T, torch.bfloat16) for T in range(1, SIMT_MAX_T + 1))
    assert not simt_bwd_fits(SIMT_MAX_T + 1, torch.bfloat16)


def test_sweep_reaches_every_branch_combination():
    """The T sweep of the GPU file reaches every value of every branch of both tensor-core launchers
    (n_tiles 1 / 2, n_left 0 / 1 / 8, NK % 32 zero and not, TMA tail boxes or none, the fp32 extra key
    or none), every combination of those that any T produces with n_left in {0, 1, 8}, and the edges of
    the CUDA-core paths; the GPU file runs each point causal and not."""
    every = {c for c in _combos(range(1, TC_FWD_MAX_T + 1)) if c[1] in (0, 1, 8)}
    missing = every - _combos(SWEEP_T)
    assert not missing, f"T sweep misses tensor-core forward branch combinations {sorted(missing)}"
    bwd = {(b["n_tiles"], b["rows0"] < 128, b["rows1"] % 32 == 0 if b["rows1"] else None, b["tail_rows"] > 0)
           for b in map(tc_bwd_branches, range(1, 257))}
    got = {(b["n_tiles"], b["rows0"] < 128, b["rows1"] % 32 == 0 if b["rows1"] else None, b["tail_rows"] > 0)
           for b in map(tc_bwd_branches, [T for T in SWEEP_T if T <= 256])}
    assert bwd == got, sorted(bwd - got)
    for T in (1, 203, 204, 256, 257, 258, SIMT_MAX_T):
        assert T in SWEEP_T


@pytest.mark.parametrize("T,causal", list(itertools.product([1, 16, 77, 129, 136, 197, 256, 257, 288], [False, True])))
def test_spikes_hold_the_mass_they_claim(T, causal):
    B, H = 2, 3
    pairs = spike_pairs(T, causal)
    rows = {r for r, _ in pairs}
    keys = {j for _, j in pairs}
    assert {i for i in (0, 127, 128, 255, 256, T - 1) if i < T} <= rows
    assert {i for i in (0, 15, 16, 127, 128, 256, T - 1) if i < T} <= keys
    if T <= TC_FWD_MAX_T and tc_fwd_branches(T)["NK"] <= T:
        assert tc_fwd_branches(T)["NK"] - 1 in keys
    qkv = spiked_qkv(B, T, H, pairs, seed=T)
    assert qkv.dtype == torch.bfloat16 and qkv.shape == (B * T, 3 * H * 64)
    p = softmax_mass(qkv, B, T, H, causal)
    for r, j in pairs:
        assert float(p[:, :, r, j].min()) > 0.9, (r, j, float(p[:, :, r, j].min()))
