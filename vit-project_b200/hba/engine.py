"""Host-side engine of the CLIP-HBA forward / live-sub-graph backward on libhba (sm_100a).

The engine owns nothing numerical: it stages the frozen weights once as bf16 (hi[/lo]) GEMM
operands, owns the HBM workspaces, and sequences C-ABI calls on the current CUDA stream.

What is computed (equal to the reference graph reached through CLIPHBA.forward, NEW:287-304, up to
fp32 re-association):
  * vision tower: conv1-as-GEMM, cls/pos, ln_pre, L residual attention blocks, ln_post, proj;
    the LAST block is evaluated for the CLS query row only (its other rows feed nothing);
  * text tower: embedding, L_t causal blocks; after the last attention only the EOT rows are kept
    (everything after it is row-wise);
  * cosine logits  exp(logit_scale) * <img, txt>.
Each tower has one live range, blocks [first, L) with first = L - n_live: the first adapted block, and
at least the last 2 vision / last 1 text blocks - the reference drivers' placement (NEW:484-544, BDRV:28-30).
Blocks below it are frozen and run in place (or come from the trunk / text cache), blocks [first, L-1)
run on all rows and keep only what the backward reads, the last block runs on the CLS / EOT rows.
Backward covers exactly the sub-graph that reaches trainable parameters: the last block's rows, then
down through the live blocks to the lowest trainable adapter.  It returns dL/dW of the adapters'
`out_proj.weight` tensors; the DoRA chain rule on top is hba.dora (fused) or plain autograd when the
reference's own DoRALayer is used.

Precision modes (hba.set_precision):
  "bf16": bf16 operands, fp32 accumulate (tcgen05 kind::f16), fp32 residual stream / LN / softmax
  "fp32": every GEMM runs three bf16 passes over hi/lo split operands (~2^-16 relative error),
          attention in exact fp32 — the parity mode (1e-3 relative vs the fp32 reference)
"""
from __future__ import annotations

import os

import torch

from . import ops
from .ops import Operand, HBA_ACT_NONE, HBA_ACT_QUICKGELU, HBA_ACT_QUICKGELU_GRAD

_PRECISION = os.environ.get("HBA_PRECISION", "bf16")
LN_EPS = 1e-5


def set_precision(mode: str):
    global _PRECISION
    if mode not in ("bf16", "fp32"):
        raise ValueError("precision must be 'bf16' or 'fp32'")
    _PRECISION = mode


def get_precision() -> str:
    return _PRECISION


def _roundup(v, m):
    return (v + m - 1) // m * m


class _Block:
    """Staged operands of one residual attention block."""
    __slots__ = ("ln1_w", "ln1_b", "ln2_w", "ln2_b", "w_in", "b_in", "w_out", "b_out", "w_fc",
                 "b_fc", "w_proj", "b_proj", "w_in_t", "w_fc_t", "w_proj_t", "w_out_t", "adapter")


class _Tower:
    __slots__ = ("blocks", "d", "heads", "T", "causal", "n_live")


class LossRequest:
    """Asks the next forward pass to fuse nn.MSELoss(reduction='mean') (BDRV:31, applied NEW:994 / NEW:597) and
    the loop's per-batch bookkeeping into the head kernel (hba_cos_mse_fwd): `target` [B, S] fp32; optional
    device scalars `bad_step` (int32, non-finite loss -> the optimiser skips the update, NEW:989-998),
    `bad_total` (int32 running count) and `total` (float64 running sum of loss * batch, NEW:1003-1004)."""
    __slots__ = ("target", "bad_step", "bad_total", "total")

    def __init__(self, target, bad_step=None, bad_total=None, total=None):
        self.target, self.bad_step, self.bad_total, self.total = target, bad_step, bad_total, total


class Engine:
    def __init__(self, model):
        self.model = model
        self.device = None
        self.precision = None
        self._bufs = {}
        self._stamp = None
        self.cache_text = True
        self.trunk_cache = None   # TrunkCache: frozen-trunk activations per image id (exact reuse)
        self.batch_ids = None     # image ids of the next forward batch (consumed by run_forward)
        self.loss_request = None  # LossRequest of the next forward batch (consumed by run_forward)
        self.loss_out = None      # the fused loss of the last forward that carried a LossRequest
        self._text_cache = None
        self._gen = 0

    # ---------------------------------------------------------------- staging
    @property
    def split(self):
        return self.precision == "fp32"

    def _param_stamp(self, rescan=False):
        # frozen tensors only: trainable adapter parameters are read live on every call.  The tensor lists
        # are collected when the weights are staged (and again whenever the adapter slots change): walking
        # the 450-parameter module tree on every forward cost 0.6 ms of host time per step.
        slots_now = tuple(id(blk.attn.out_proj) for tower in (self.model.visual.transformer, self.model.transformer)
                          for blk in tower.resblocks)
        if rescan or getattr(self, "_stamp_slots", None) != slots_now:
            self._stamp_slots = slots_now
            self._stamp_params = [p for p in self.model.parameters() if not p.requires_grad]
            self._stamp_buffers = list(self.model.buffers())
        stamp = sum(p._version for p in self._stamp_params) + 7919 * sum(b._version for b in self._stamp_buffers)
        # which out_proj slots hold adapters is part of the staging (module surgery restages)
        slots = tuple(id(blk.attn.out_proj.original_layer) if hasattr(blk.attn.out_proj, "original_layer")
                      else -id(blk.attn.out_proj)
                      for tower in (self.model.visual.transformer, self.model.transformer)
                      for blk in tower.resblocks)
        return (stamp, slots)

    def _operand(self, W, K_pad=None, transpose=False):
        W = W.detach()
        if W.dtype != torch.float32:
            W = W.float()
        W = W.contiguous()
        rows, cols = W.shape
        if transpose:
            op = Operand.empty(cols, rows if K_pad is None else K_pad, self.split, W.device,
                               zero=K_pad is not None)
        else:
            op = Operand.empty(rows, cols if K_pad is None else K_pad, self.split, W.device,
                               zero=K_pad is not None)
        ops.split_bf16(W, op, transpose=transpose)
        return op

    @staticmethod
    def _live_blocks(resblocks, n_default):
        """Blocks from the first adapted one to the end (at least the `n_default` of the reference drivers' placement,
        BDRV:28-30: the staging - and with it every kernel launch - of that placement is unchanged)."""
        first = next((i for i, blk in enumerate(resblocks) if not isinstance(blk.attn.out_proj, torch.nn.Linear)),
                     len(resblocks))
        return max(n_default, len(resblocks) - first)

    def _stage_tower(self, resblocks, T, causal, n_default):
        n_live = min(len(resblocks), self._live_blocks(resblocks, n_default))
        first_adapter = next((i for i, blk in enumerate(resblocks) if not isinstance(blk.attn.out_proj, torch.nn.Linear)),
                             len(resblocks))
        tw = _Tower()
        tw.blocks, tw.T, tw.causal = [], T, causal
        L = len(resblocks)
        for i, blk in enumerate(resblocks):
            b = _Block()
            attn = blk.attn
            b.ln1_w, b.ln1_b = blk.ln_1.weight.detach(), blk.ln_1.bias.detach()
            b.ln2_w, b.ln2_b = blk.ln_2.weight.detach(), blk.ln_2.bias.detach()
            b.w_in, b.b_in = self._operand(attn.in_proj_weight), attn.in_proj_bias.detach()
            op = attn.out_proj
            b.adapter = not isinstance(op, torch.nn.Linear)
            if b.adapter:
                b.w_out, b.b_out = None, None  # supplied per call (the adapter's .weight / .bias)
            else:
                if op.weight.requires_grad:
                    raise RuntimeError("libhba: a plain out_proj.weight requires grad; only adapter "
                                       "modules (DoRA) on out_proj are trainable on this path")
                b.w_out, b.b_out = self._operand(op.weight), op.bias.detach()
            b.w_fc, b.b_fc = self._operand(blk.mlp.c_fc.weight), blk.mlp.c_fc.bias.detach()
            b.w_proj, b.b_proj = self._operand(blk.mlp.c_proj.weight), blk.mlp.c_proj.bias.detach()
            live = i >= L - n_live
            # (dX through a FROZEN out_proj is only ever needed when an adapter sits below it - never in the
            # placements apply_dora_to_ViT produces for the drivers' 2 + 1)
            b.w_out_t = (self._operand(op.weight, transpose=True)
                         if live and not b.adapter and i > first_adapter else None)
            b.w_in_t = self._operand(attn.in_proj_weight, transpose=True) if live else None
            b.w_fc_t = self._operand(blk.mlp.c_fc.weight, transpose=True) if live else None
            b.w_proj_t = self._operand(blk.mlp.c_proj.weight, transpose=True) if live else None
            tw.blocks.append(b)
        tw.n_live = n_live
        tw.d = resblocks[0].attn.embed_dim
        tw.heads = resblocks[0].attn.num_heads
        if tw.d // tw.heads != 64:
            raise RuntimeError("libhba: head_dim must be 64")
        return tw

    def prepare(self, device):
        """(Re)stages every frozen weight on `device` in the current precision mode."""
        m = self.model
        self.device, self.precision = device, _PRECISION
        for p in list(m.parameters()) + list(m.buffers()):
            if p.device != device:
                raise RuntimeError("libhba: move the model to the CUDA device before calling it")
        v = m.visual
        self.P = v.conv1.weight.shape[-1]
        self.res = v.input_resolution
        self.grid = self.res // self.P
        self.vis = self._stage_tower(v.transformer.resblocks, self.grid ** 2 + 1, False, 2)
        d = self.vis.d
        self.kp = _roundup(3 * self.P * self.P, 64)
        self.w_conv = self._operand(v.conv1.weight.detach().reshape(d, -1), K_pad=self.kp)
        self.cls, self.pos = v.class_embedding.detach(), v.positional_embedding.detach()
        self._pos_cache = {}
        self.ln_pre = (v.ln_pre.weight.detach(), v.ln_pre.bias.detach())
        self.ln_post = (v.ln_post.weight.detach(), v.ln_post.bias.detach())
        self.proj_t = self._operand(v.proj, transpose=True)   # [E, d]: B operand of x @ proj
        self.proj_n = self._operand(v.proj)                   # [d, E]: B operand of g @ proj^T
        self.txt = self._stage_tower(m.transformer.resblocks, m.context_length, True, 1)
        self.tok_table = m.token_embedding.weight.detach()
        self.tpos = m.positional_embedding.detach()
        self.ln_final = (m.ln_final.weight.detach(), m.ln_final.bias.detach())
        self.tproj_t = self._operand(m.text_projection, transpose=True)
        self.tproj_n = self._operand(m.text_projection)
        self.E = m.text_projection.shape[1]
        self.logit_scale = m.logit_scale.detach().reshape(1)
        self._bufs.clear()
        self._text_cache = None
        self._stamp = self._param_stamp(rescan=True)

    def ensure(self, device):
        if (self.device != device or self.precision != _PRECISION
                or self._stamp != self._param_stamp()):
            self.prepare(device)

    # ---------------------------------------------------------------- workspaces
    def _buf(self, name, shape, dtype=torch.float32, zero=False):
        key = (name, tuple(shape), dtype)
        t = self._bufs.get(key)
        if t is None:
            t = (torch.zeros if zero else torch.empty)(*shape, dtype=dtype, device=self.device)
            self._bufs[key] = t
        return t

    def _opbuf(self, name, rows, K, zero=False):
        width = 2 * K if self.split else K
        return Operand(self._buf(name, (rows, width), torch.bfloat16, zero=zero), rows, K,
                       K if self.split else 0)

    def _positional(self, grid_now):
        if grid_now == self.grid:
            return self.pos
        if grid_now not in self._pos_cache:
            # CLIP-HBA `pos_embedding=True`: bicubic resize of the patch part of the table
            # (one-off weight preparation, identity at the native 224^2 resolution)
            g = self.grid
            patch = self.pos[1:].reshape(1, g, g, -1).permute(0, 3, 1, 2)
            patch = torch.nn.functional.interpolate(patch, size=(grid_now, grid_now), mode="bicubic",
                                                    align_corners=False)
            patch = patch.permute(0, 2, 3, 1).reshape(grid_now * grid_now, -1)
            self._pos_cache[grid_now] = torch.cat([self.pos[:1], patch], 0).contiguous()
        return self._pos_cache[grid_now]

    # ---------------------------------------------------------------- building blocks
    def _act_dtype(self):
        """dtype of the kept qkv / MLP pre-activations and of the all-row attention gradients."""
        return torch.float32 if self.split else torch.bfloat16

    def _qkv_buffer(self, tag, M, d):
        return self._buf(tag + ".qkv", (M, 3 * d), self._act_dtype())

    def _gemm_qkv(self, h, w_in, b_in, qkv, M):
        if self.split:
            ops.gemm(h, w_in, M, bias=b_in, out_f32=qkv)
        else:
            ops.gemm(h, w_in, M, bias=b_in, out=Operand(qkv, M, qkv.shape[1], 0))

    def _adapter_operands(self, W):
        """bf16 operands of an adapter weight W [out, in]: (w [out,in], wt [in,out])."""
        cached = getattr(W, "_hba_ops", None)
        if cached is not None and cached[2] == self.precision:
            return cached[0], cached[1]
        Wd = W.detach()
        out_f, in_f = Wd.shape
        w = Operand.empty(out_f, in_f, self.split, Wd.device)
        wt = Operand.empty(in_f, out_f, self.split, Wd.device)
        if Wd.t().is_contiguous():
            base = Wd.t()
            ops.split_bf16(base, w, transpose=True)
            ops.split_bf16(base, wt)
        else:
            base = Wd.contiguous()
            ops.split_bf16(base, w)
            ops.split_bf16(base, wt, transpose=True)
        return w, wt

    def _block_weights(self, blk, adapters, i, need_grad):
        """(w [out,in], wt [in,out], bias, trainable) of block i's out_proj."""
        if blk.adapter:
            W, bias = adapters[i]
            w, wt = self._adapter_operands(W)
            return w, wt, bias.detach(), bool(need_grad and W.requires_grad)
        return blk.w_out, blk.w_out_t, blk.b_out, False

    def _skinny(self, tag, R, N, K):
        """Split-K arguments of a row GEMM (R = the CLS / EOT rows, one row tile): its N / 256 output tiles would
        leave most of the 74 CTA pairs idle while a few SMs stream the whole weight matrix; split along K the
        matrix is pulled by ~74 pairs at once and the epilogue runs in the slice reduction (same fused epilogue).
        The workspace is per tag: the two towers run on different streams."""
        if R > 256:
            return {}
        s = ops.auto_k_slices(R, N, K, min_kblocks=4)
        if s <= 1:
            return {}
        return {"k_slices": s, "k_workspace": self._buf(tag + ".kws", (s * R * N,))}

    def _attn_part(self, tw, blk, tag, x_in, B, a, qkv=None, a_f32=None):
        """ln_1 -> in_proj -> softmax attention on all rows into the GEMM operand `a` (and in fp32 into `a_f32` when
        given).  `qkv` receives the projections when the attention backward reads them, else the tower's scratch."""
        T, d = tw.T, tw.d
        M = B * T
        h = self._opbuf(tag + ".h", M, d)
        ops.layernorm_fwd(x_in, M, d, blk.ln1_w, blk.ln1_b, LN_EPS, y=h)
        if qkv is None:
            qkv = self._qkv_buffer(tag, M, d)
        self._gemm_qkv(h, blk.w_in, blk.b_in, qkv, M)
        ops.attention_fwd(qkv, B, T, tw.heads, causal=tw.causal, out=a, out_f32=a_f32)

    def _live_part(self, tw, blk, tag, a, x_in, x_mid, x_out, B, w_out, b_out, h_pre=None):
        """out_proj (+ residual) -> ln_2 -> MLP (+ residual) on all rows (x_* are fp32 [M, d], possibly the same)."""
        d = tw.d
        M = B * tw.T
        ops.gemm(a, w_out, M, bias=b_out, residual=x_in, out_f32=x_mid)
        h = self._opbuf(tag + ".h", M, d)
        ops.layernorm_fwd(x_mid, M, d, blk.ln2_w, blk.ln2_b, LN_EPS, y=h)
        hid = self._opbuf(tag + ".hid", M, 4 * d)
        ops.gemm(h, blk.w_fc, M, bias=blk.b_fc, act=HBA_ACT_QUICKGELU, out=hid, pre_out=h_pre)
        ops.gemm(hid, blk.w_proj, M, bias=blk.b_proj, residual=x_mid, out_f32=x_out)

    def _frozen_blocks(self, tw, tag, x, B, upto):
        """Blocks [0, upto) in place on all rows of x (fp32 [B*T, d]): nothing below the first adapter is
        differentiated."""
        for blk in tw.blocks[:upto]:
            if blk.adapter:
                raise RuntimeError("libhba: an adapter below the staged live blocks (restage: Engine.prepare)")
            a = self._opbuf(tag + ".a", B * tw.T, tw.d)
            self._attn_part(tw, blk, tag, x, B, a)
            self._live_part(tw, blk, tag, a, x, x, x, B, blk.w_out, blk.b_out)

    def _live_blocks_fwd(self, tw, tag, x, B, adapters, need_grad, cache_ctx=None, keep_input=False):
        """Blocks [first, L-1) on all M = B*T rows, `first` = L - tw.n_live.  The backward walks them down from the top
        and stops at the lowest trainable adapter, so a block keeps
          * its qkv when the attention backward runs through it (a trainable adapter below it);
          * its MLP pre-activation, x_mid and x_out (the input of the block above) when the backward passes through
            its MLP (a trainable adapter at or below it);
          * its attention output as a GEMM operand (the dW operand) when it is trainable.
        Otherwise it runs in place on x like a frozen block - except on the input itself when `keep_input` (the text
        trunk cache).  cache_ctx: the vision trunk cache, which holds the first live block's input and attention output.
        -> (x, {block index: what its backward reads}, whether a trainable adapter sits in [first, L-1))."""
        L, d, M = len(tw.blocks), tw.d, B * tw.T
        first = L - tw.n_live
        blocks, reach = {}, False
        for i in range(first, L - 1):
            blk = tw.blocks[i]
            w, wt, bias, train = self._block_weights(blk, adapters, i, need_grad)
            below, reach = reach, reach or train
            name = f"{tag}{i}"
            # (block L-2 may leave its dW operand in the tower's scratch: no later block writes it)
            a = self._opbuf(name + ".a" if train and i < L - 2 else tag + ".a", M, d)
            qkv = None
            if i == first and cache_ctx is not None and cache_ctx["hit"]:
                a_f32 = cache_ctx["a"]
                ops.split_bf16(a_f32, a)
            else:
                fill = i == first and cache_ctx is not None
                # (the dW reads the operand `a`; a trainable block writes the fp32 copy all the same)
                a_f32 = self._keep(name + ".a_f32", (M, d)) if train or fill else None
                if below:
                    qkv = self._keep(name + ".qkv", (M, 3 * d), self._act_dtype())
                self._attn_part(tw, blk, tag, x, B, a, qkv, a_f32)
                if fill:
                    cache_ctx["cache"].store(cache_ctx["ids"], x, a_f32)
            x_mid = self._keep(name + ".x_mid", (M, d)) if reach or (keep_input and i == first) else x
            x_out = self._keep(name + ".x_out", (M, d)) if reach else x_mid
            h_pre = self._keep(name + ".h_pre", (M, 4 * d), self._act_dtype()) if reach else None
            self._live_part(tw, blk, tag, a, x, x_mid, x_out, B, w, bias, h_pre)
            if reach:
                blocks[i] = {"train": train, "below": below, "a_op": a, "qkv": qkv, "x_in": x, "x_mid": x_mid,
                             "h_pre": h_pre, "wt": wt}
            x = x_out
        return x, blocks, reach

    def _last_block_keep(self, tag, R, d, train, below, x_in, wt):
        """What the backward reads of the last block's R rows - None when no gradient passes through it."""
        if not (train or below):
            return None
        return {"x_mid": self._keep(tag + ".xmidZ", (R, d)), "x_out": self._keep(tag + ".xoutZ", (R, d)),
                "h_pre": self._keep(tag + ".hpreZ", (R, 4 * d), self._act_dtype()), "x_in": x_in, "wt": wt}

    def _last_rows(self, tw, tag, a_rows, x_rows, R, w_out, b_out, keep, ln, proj_t):
        """out_proj + MLP of the last block on R selected rows (CLS rows / EOT rows), then the final LN and the
        projection.  a_rows: Operand [R, d] (attention output rows); x_rows: fp32 view [R, *] of the block input rows
        (row stride arbitrary).  Returns the features [R, E] fp32."""
        blk, d = tw.blocks[-1], tw.d
        x_mid = keep["x_mid"] if keep else self._buf(tag + ".xmid", (R, d))
        ops.gemm(a_rows, w_out, R, bias=b_out, residual=x_rows, out_f32=x_mid, **self._skinny(tag, R, d, d))
        h = self._opbuf(tag + ".h2", max(R, 128), d)
        ops.layernorm_fwd(x_mid, R, d, blk.ln2_w, blk.ln2_b, LN_EPS, y=h)
        hid = self._opbuf(tag + ".hid2", max(R, 128), 4 * d)
        ops.gemm(h, blk.w_fc, R, bias=blk.b_fc, act=HBA_ACT_QUICKGELU, out=hid,
                 pre_out=keep["h_pre"] if keep else None, **self._skinny(tag, R, 4 * d, d))
        x_out = keep["x_out"] if keep else self._buf(tag + ".xout", (R, d))
        ops.gemm(hid, blk.w_proj, R, bias=blk.b_proj, residual=x_mid, out_f32=x_out,
                 **self._skinny(tag, R, d, 4 * d))
        hp = self._opbuf(tag + ".lnf", max(R, 128), d)
        ops.layernorm_fwd(x_out, R, d, ln[0], ln[1], LN_EPS, y=hp)
        feat = self._keep(tag + ".feat", (R, self.E))
        ops.gemm(hp, proj_t, R, out_f32=feat, **self._skinny(tag, R, self.E, d))
        return feat

    # ---------------------------------------------------------------- forward
    def _keep(self, name, shape, dtype=torch.float32):
        return self._buf("keep." + name, shape, dtype)

    def vision_trunk(self, images, upto):
        """conv1 + cls/pos + ln_pre + blocks [0, upto) on all rows. Returns x fp32 [B*T, d]."""
        B = images.shape[0]
        if images.shape[2] % self.P or images.shape[3] % self.P or images.shape[2] != images.shape[3]:
            raise RuntimeError("libhba: image side must be a multiple of the patch size and square")
        grid = images.shape[2] // self.P
        tw = self.vis
        if grid != self.grid:
            if not self._pos_flag:
                raise RuntimeError("libhba: image resolution differs from the model's and "
                                   "pos_embedding=False")
            tw = _Tower()
            tw.blocks, tw.d, tw.heads, tw.causal = self.vis.blocks, self.vis.d, self.vis.heads, False
            tw.n_live = self.vis.n_live
            tw.T = grid * grid + 1
        npatch, d, T = grid * grid, tw.d, tw.T
        M = B * T
        images = images.contiguous().float()
        patches = self._opbuf("v.patches", max(B * npatch, 128), self.kp, zero=True)
        ops.im2col_patches(images, self.P, patches)
        conv = self._buf("v.conv", (B * npatch, d))
        ops.gemm(patches, self.w_conv, B * npatch, out_f32=conv)
        x = self._buf("v.x", (M, d))
        ops.assemble_tokens_ln(conv, B, npatch, d, self.cls, self._positional(grid), self.ln_pre[0],
                               self.ln_pre[1], LN_EPS, x)
        self._frozen_blocks(tw, "v", x, B, upto)
        return x, tw

    def vision_head(self, x, tw, B, adapters, need_grad, cache_ctx=None):
        """Live blocks [first, L-1) on all rows (x: their input), block L-1 for the CLS query rows, ln_post, proj.
        `adapters` maps block index -> (W, bias) for adapter blocks.  Returns (img_feat [B,E] fp32, saved dict)."""
        L, T, d = len(tw.blocks), tw.T, tw.d
        M = B * T
        if tw.n_live > 2 and self.split and T > 200:
            raise NotImplementedError("libhba fp32 mode: more than two adapted vision blocks need the full attention "
                                      "backward, whose fp32 form holds T <= 200 tokens (use the bf16 mode)")
        x, blocks, below = self._live_blocks_fwd(tw, "v", x, B, adapters, need_grad, cache_ctx)
        blk = tw.blocks[L - 1]
        w, wt, bias, train = self._block_weights(blk, adapters, L - 1, need_grad)
        keep = self._last_block_keep("v", B, d, train, below, x, wt)
        h = self._opbuf("v.h", M, d)
        ops.layernorm_fwd(x, M, d, blk.ln1_w, blk.ln1_b, LN_EPS, y=h)
        qkv = self._keep("v.qkvZ", (M, 3 * d), self._act_dtype()) if below else self._qkv_buffer("v", M, d)
        self._gemm_qkv(h, blk.w_in, blk.b_in, qkv, M)
        a_cls = self._opbuf("v.acls", max(B, 128), d)
        a_f32 = self._keep("v.aZ", (B, d)) if keep else None
        ops.attention_fwd(qkv, B, T, tw.heads, first_row_only=True, out=a_cls, out_f32=a_f32)
        x_cls = x.view(B, T * d)[:, :d]  # CLS rows of the block input, row stride T*d
        feat = self._last_rows(tw, "v", a_cls, x_cls, B, w, bias, keep, self.ln_post, self.proj_t)
        if keep:
            keep.update(a_f32=a_f32, qkv=qkv)
        return feat, {"tw": tw, "R": B, "blocks": blocks, "below": below, "trainZ": train, "keepZ": keep}

    def _eot_attention(self, x, eot, S, qkv=None):
        """ln_1 -> in_proj -> causal attention of the last text block on all rows, then the EOT rows of its output and
        of its input.  -> (attention operand, attention fp32, block input), each [S, d]."""
        tw = self.txt
        M, d, blk = S * tw.T, tw.d, tw.blocks[-1]
        h = self._opbuf("t.h", M, d)
        ops.layernorm_fwd(x, M, d, blk.ln1_w, blk.ln1_b, LN_EPS, y=h)
        if qkv is None:
            qkv = self._qkv_buffer("t", M, d)
        self._gemm_qkv(h, blk.w_in, blk.b_in, qkv, M)
        a_all = self._buf("t.a_f32", (M, d))
        ops.attention_fwd(qkv, S, tw.T, tw.heads, causal=True, out_f32=a_all)
        # (persistent buffers, not fresh tensors: they are produced on the side stream and read by
        # the backward pass on the main stream - nothing here may be recycled by the caching allocator)
        a_eot = self._buf("t.a_eot", (S, d))
        x_eot = self._buf("t.x_eot", (S, d))
        ops.gather_rows(a_all, eot, d, a_eot)
        ops.gather_rows(x, eot, d, x_eot)
        a_op = self._opbuf("t.a_op", max(S, 128), d, zero=True)
        ops.split_bf16(a_eot, a_op)
        return a_op, a_eot, x_eot

    def text_features(self, tokens, adapters, need_grad):
        """Text tower -> (txt_feat [S, E], saved dict).  Everything frozen is cached per token tensor (the prompts never
        change, NEW:282): blocks [0, first) and, when only the last block is live, its attention and EOT rows too.
        Blocks [first, L-1) run on all S*T rows; after the last attention only the EOT rows are kept."""
        tw = self.txt
        S, T = tokens.shape
        d, L = tw.d, len(tw.blocks)
        first = L - tw.n_live
        key = (tokens.data_ptr(), tokens._version, S, T, first)
        cache = self._text_cache if (self.cache_text and self._text_cache
                                     and self._text_cache["key"] == key) else None
        if cache is None:
            x = self._buf("t.x", (S * T, d))
            ops.embed_tokens(tokens, self.tok_table, self.tpos, x)
            self._frozen_blocks(tw, "t", x, S, first)
            eot = (tokens.argmax(dim=-1) + torch.arange(S, device=tokens.device) * T).contiguous()
            # (the entry keeps the token tensor alive: the key holds its ADDRESS, and the caching allocator would hand
            # the address of a freed prompt tensor to the next model's prompts - other class names, same key)
            cache = {"key": key, "x": x, "eot": eot, "tokens": tokens}
            if first == L - 1:
                cache["rows"] = self._eot_attention(x, eot, S)
            if self.cache_text:
                self._text_cache = cache
        x, blocks, below = self._live_blocks_fwd(tw, "t", cache["x"], S, adapters, need_grad, keep_input=True)
        qkv = self._keep("t.qkvZ", (S * T, 3 * d), self._act_dtype()) if below else None
        a_op, a_eot, x_eot = cache["rows"] if "rows" in cache else self._eot_attention(x, cache["eot"], S, qkv)
        blk = tw.blocks[L - 1]
        w, wt, bias, train = self._block_weights(blk, adapters, L - 1, need_grad)
        keep = self._last_block_keep("t", S, d, train, below, x, wt)
        feat = self._last_rows(tw, "t", a_op, x_eot, S, w, bias, keep, self.ln_final, self.tproj_t)
        if keep:
            keep.update(a_f32=a_eot, qkv=qkv)
        return feat, {"tw": tw, "R": S, "blocks": blocks, "below": below, "trainZ": train, "keepZ": keep,
                      "eot": cache["eot"]}

    def _side_stream(self):
        st = self.__dict__.get("_side")
        if st is None or st.device != self.device:
            st = self.__dict__["_side"] = torch.cuda.Stream(device=self.device)
        return st

    def run_forward(self, images, tokens, pos_embedding, v_adapters, t_adapters, need_grad):
        """-> (pred [B, S] fp32 (fresh tensor), saved state for run_backward)."""
        self.ensure(images.device)
        self._pos_flag = bool(pos_embedding)
        tokens = tokens.reshape(-1, tokens.shape[-1])
        if tokens.dtype != torch.int64:
            tokens = tokens.long()
        tokens = tokens if tokens.is_contiguous() else tokens.contiguous()
        B = images.shape[0]
        L = len(self.vis.blocks)
        ids, self.batch_ids = self.batch_ids, None
        req, self.loss_request = self.loss_request, None
        if req is not None:
            t = req.target
            if (t.dtype != torch.float32 or not t.is_contiguous() or t.device != images.device
                    or t.ndim != 2 or t.shape[0] != B or t.shape[1] != tokens.shape[0]):
                raise RuntimeError("libhba: fused MSE needs contiguous fp32 targets of shape [batch, prompts] "
                                   "on the model's device")
        cache_ctx = None
        native = images.shape[2] == self.res and images.shape[3] == self.res
        if self.trunk_cache is not None and ids is not None and L >= 2 and native:
            if len(ids) != B:
                raise RuntimeError("libhba: batch_ids does not match the image batch")
            if isinstance(ids, torch.Tensor):
                cache_ctx = self.trunk_cache.lookup_device_ids(self, ids)
            else:
                cache_ctx = self.trunk_cache.lookup(self, ids)
        # The two towers are independent until the cosine head: the text tower (small persistent kernels,
        # 2.4 waves of tiles per GEMM at 66 x 77 rows) is enqueued on a side stream so that its kernels
        # fill the SMs the vision tower's kernel tails leave idle, and vice versa.  Same kernels, same
        # arguments: results are unchanged.  Fork / join are stream events, so the pair is captured into a
        # CUDA graph as two parallel branches.  HBA_TEXT_STREAM=0 keeps everything on one stream.
        side = None
        if os.environ.get("HBA_TEXT_STREAM", "1") != "0":
            main = torch.cuda.current_stream(self.device)
            side = self._side_stream()
            side.wait_stream(main)    # fork: the adapters' merged weights were produced on the main stream
            with torch.cuda.stream(side):
                txt_feat, st = self.text_features(tokens, t_adapters, need_grad)
        if cache_ctx is not None and cache_ctx["hit"]:
            x, tw = cache_ctx["x"], self.vis
        else:
            x, tw = self.vision_trunk(images, L - self.vis.n_live)
        img_feat, sv = self.vision_head(x, tw, B, v_adapters, need_grad, cache_ctx)
        if side is None:
            txt_feat, st = self.text_features(tokens, t_adapters, need_grad)
        else:
            main.wait_stream(side)   # join: the cosine head needs both towers
        pred = torch.empty(B, txt_feat.shape[0], device=self.device)
        loss = None
        if req is None:
            ops.cos_head_fwd(img_feat, txt_feat, self.logit_scale, pred)
        else:
            loss = torch.empty((), device=self.device)
            ops.cos_mse_fwd(img_feat, txt_feat, self.logit_scale, pred, B=B, target=req.target, loss=loss,
                            bad_step=req.bad_step, bad_total=req.bad_total, total=req.total,
                            workspace=self._buf("head.ws", (B + 1,), zero=True))
        self._gen += 1
        return pred, {"v": sv, "t": st, "img_feat": img_feat, "txt_feat": txt_feat, "gen": self._gen,
                      "loss": loss, "pred": pred.detach(), "target": req.target if req is not None else None}

    # ---------------------------------------------------------------- backward
    def _grad_operand(self, name, g, rows, cols, transpose=False, k_pad=None):
        """fp32 gradient [rows, cols] -> bf16 operand ([rows, cols] or, transposed, [cols, k_pad])."""
        if transpose:
            op = self._opbuf(name, cols, k_pad, zero=True)
            ops.split_bf16(g[:rows], op, transpose=True)
        else:
            op = self._opbuf(name, max(rows, 128), cols)
            ops.split_bf16(g[:rows], op)
        return op

    def _mlp_rows_bwd(self, blk, tag, dxo, R, d, h_pre, x_mid):
        """dxo [R, d] holds dL/dx_out; on return it holds dL/dx_mid (MLP + LN2 + residual)."""
        g1 = self._grad_operand(tag + ".g1", dxo, R, d)
        gh = self._opbuf(tag + ".gh", max(R, 128), 4 * d)
        ops.gemm(g1, blk.w_proj_t, R, act=HBA_ACT_QUICKGELU_GRAD, aux=h_pre, out=gh, **self._skinny(tag, R, 4 * d, d))
        d_ln2 = self._buf(tag + ".dln2", (R, d))
        ops.gemm(gh, blk.w_fc_t, R, out_f32=d_ln2, **self._skinny(tag, R, d, 4 * d))
        ops.layernorm_bwd(d_ln2, x_mid, R, d, blk.ln2_w, LN_EPS, dxo, accumulate=True)

    def _dw(self, tag, dY, a_f32, R, d_out, d_in, a_op=None):
        """dW[out, in] = sum_r dY[r, out] a[r, in]: both operands are read MN-major (as [K = rows, M / N]
        matrices, no transposition pass; rows beyond R are zero-filled by TMA) and the K = R rows are split
        into slices when the 16 output tiles of a 1024 x 1024 gradient would leave 58 of 74 CTA pairs idle."""
        A = self._grad_operand(f"{tag}.dy{R}", dY, R, d_out)
        # (a_op: the forward pass' own bf16 operand of the same activation - identical to restaging a_f32)
        Bo = a_op if a_op is not None else self._grad_operand(f"{tag}.a{R}", a_f32, R, d_in)
        dW = torch.empty(d_out, d_in, device=self.device)
        s = ops.auto_k_slices(d_out, d_in, R)
        ws = self._buf("b.k_ws", (s * d_out * d_in,)) if s > 1 else None
        ops.gemm(Operand(A.buf, R, d_out, A.lo_off), Operand(Bo.buf, R, d_in, Bo.lo_off), a_mn=True, b_mn=True,
                 K=R, out_f32=dW, k_slices=s, k_workspace=ws)
        return dW

    def run_backward(self, saved, d_pred, d_loss=None):
        """-> dict {('v', block_index) | ('t', block_index): dL/dW [out, in] fp32}.
        d_loss: upstream gradient of the fused loss (LossRequest); with d_pred None the head backward reads
        (pred, target) directly (hba_cos_mse_bwd) and no dL/dpred tensor is ever formed."""
        if saved["gen"] != self._gen:
            raise RuntimeError("libhba: backward called after a newer forward pass overwrote the "
                               "saved activations (call backward before the next forward)")
        grads = {}
        img_feat, txt_feat = saved["img_feat"], saved["txt_feat"]
        B, S, E = img_feat.shape[0], txt_feat.shape[0], self.E
        d_img = self._buf("b.dimg", (B, E))
        d_txt = self._buf("b.dtxt", (S, E))
        if d_loss is not None and d_pred is None:
            ops.cos_mse_bwd(img_feat, txt_feat, self.logit_scale, saved["pred"], saved["target"], d_img, d_txt,
                            B=B, d_loss=d_loss.reshape(1).float())
        else:
            if d_loss is not None:   # both outputs were used downstream: fold the loss gradient into dL/dpred
                d_pred = d_pred + (2.0 / saved["pred"].numel()) * d_loss * (saved["pred"] - saved["target"])
            ops.cos_head_bwd(img_feat, txt_feat, self.logit_scale, d_img, d_txt,
                             d_pred=d_pred.contiguous().float())
        self._tower_bwd("t", saved["t"], d_txt, grads)
        self._tower_bwd("v", saved["v"], d_img, grads)
        return grads

    def _tower_bwd(self, side, s, d_feat, grads):
        """Backward of one tower from dL/d(features): projection, final LN and MLP of the last block on its R rows (CLS
        / EOT rows) and its out_proj dW; then, when a trainable adapter sits below, out_proj dX, the last attention's
        backward onto all rows of its input, and the walk down the live full blocks."""
        if not (s["trainZ"] or s["below"]):
            return
        tw, R, kz = s["tw"], s["R"], s["keepZ"]
        L, d, T, H = len(tw.blocks), tw.d, tw.T, tw.heads
        M = R * T
        blk, tag = tw.blocks[L - 1], side + "b"
        ln, proj_n = (self.ln_post, self.proj_n) if side == "v" else (self.ln_final, self.tproj_n)
        g = self._grad_operand(tag + ".g0", d_feat, R, self.E)
        d_ln = self._buf(tag + ".dln", (R, d))
        ops.gemm(g, proj_n, R, out_f32=d_ln, **self._skinny(tag, R, d, self.E))
        dxo = self._buf(tag + ".dxo", (R, d))
        ops.layernorm_bwd(d_ln, kz["x_out"], R, d, ln[0], LN_EPS, dxo)
        self._mlp_rows_bwd(blk, tag, dxo, R, d, kz["h_pre"], kz["x_mid"])   # dxo := dL/d(out_proj output) of the rows
        if s["trainZ"]:
            grads[(side, L - 1)] = self._dw(tag, dxo, kz["a_f32"], R, d, d)
        if not s["below"]:
            return
        wt = kz["wt"] if kz["wt"] is not None else self._frozen_wt(blk)
        g2 = self._grad_operand(tag + ".g2", dxo, R, d)
        d_a = self._buf(tag + ".da", (R, d))
        ops.gemm(g2, wt, R, out_f32=d_a, **self._skinny(tag, R, d, d))
        if side == "v":   # only the CLS query rows were attended from
            d_qkv = self._buf(tag + ".dqkv", (M, 3 * d))
            ops.attention_bwd_row0(kz["qkv"], R, T, H, d_a, d_qkv)
            gq = self._grad_operand(tag + ".gq", d_qkv, M, 3 * d)
        else:             # the causal attention of every row, with a zero gradient outside the EOT rows
            dt = self._act_dtype()
            d_a_all = self._buf(tag + ".da_all", (M, d), dt)
            d_a_all.zero_()
            d_a_all.index_copy_(0, s["eot"], d_a.to(dt))
            d_qkv = self._buf(tag + ".dqkv", (M, 3 * d), dt)
            ops.attention_bwd(kz["qkv"], R, T, H, d_a_all, d_qkv, causal=True)
            gq = self._grad_operand(tag + ".gq", d_qkv, M, 3 * d) if self.split else Operand(d_qkv, M, 3 * d, 0)
        d_ln1 = self._buf(tag + ".dln1", (M, d))
        ops.gemm(gq, blk.w_in_t, M, out_f32=d_ln1)
        dx = self._buf(tag + ".dx", (M, d))
        ops.layernorm_bwd(d_ln1, kz["x_in"], M, d, blk.ln1_w, LN_EPS, dx)
        # residual path of the CLS / EOT rows
        if side == "v":
            ops.add_rows(dx, dxo, R, d, dst_row_step=T)
        else:
            dx.index_add_(0, s["eot"], dxo)
        self._blocks_bwd(tw, side, s["blocks"], dx, R, grads)

    def _blocks_bwd(self, tw, side, blocks, dx, B, grads):
        """dx [M, d] = dL/d(output of block L-2) on entry.  Walks the live full blocks down, collecting dL/dW of every
        trainable out_proj, and stops at the lowest trainable adapter."""
        L, d, T, H = len(tw.blocks), tw.d, tw.T, tw.heads
        M = B * T
        for i in range(L - 2, -1, -1):
            blk, kp = tw.blocks[i], blocks[i]
            tag = f"{side}bg{i}"
            self._mlp_rows_bwd(blk, tag, dx, M, d, kp["h_pre"], kp["x_mid"])       # dx := dL/d(out_proj output)
            if kp["train"]:
                grads[(side, i)] = self._dw(tag, dx, None, M, d, d, a_op=kp["a_op"])
            if not kp["below"]:
                break
            g = self._grad_operand(tag + ".gy", dx, M, d)
            d_a = self._buf(tag + ".da", (M, d), self._act_dtype())   # (bf16 mode: the all-bf16 form of hba_attention_bwd)
            if self.split:
                ops.gemm(g, kp["wt"], M, out_f32=d_a)
            else:
                ops.gemm(g, kp["wt"], M, out=Operand(d_a, M, d, 0))
            d_qkv = self._buf(tag + ".dqkv", (M, 3 * d), self._act_dtype())
            ops.attention_bwd(kp["qkv"], B, T, H, d_a, d_qkv, causal=tw.causal)
            gq = self._grad_operand(tag + ".gq", d_qkv, M, 3 * d) if self.split else Operand(d_qkv, M, 3 * d, 0)
            d_ln1 = self._buf(tag + ".dln1", (M, d))
            ops.gemm(gq, blk.w_in_t, M, out_f32=d_ln1)
            # residual: dL/dx_in = dL/d(out_proj output) + ln_1 backward of the attention branch
            ops.layernorm_bwd(d_ln1, kp["x_in"], M, d, blk.ln1_w, LN_EPS, dx, accumulate=True)

    def _frozen_wt(self, blk):
        if getattr(blk, "w_out_t", None) is not None:
            return blk.w_out_t
        raise RuntimeError("libhba: backward through a frozen out_proj of the last block is not "
                           "staged (adapter expected on the last block)")


class TrunkCache:
    """HBM cache of the frozen vision trunk per image: the input of the first live block (`first`, L-2 in the
    reference drivers' placement) and that block's attention output (ln_1 -> in_proj -> attention is
    frozen-on-frozen there), both fp32.

    Exactness: train images are never augmented (NEW:183-188) and blocks below `first` plus the attention
    half of block `first` hold no trainable parameter (NEW:665-669), so for an un-perturbed image these
    activations are identical in every epoch; the cached path runs the same kernels on the same
    values and is bit-identical to recomputation.  Callers must not pass ids for perturbed images
    (`image_noise`, `uniform_images` windows, NEW:880-916)."""

    def __init__(self, capacity):
        self.capacity = capacity
        self.x = self.a = None
        self.present = set()
        self.stamp = None

    @staticmethod
    def _stamp_of(eng):
        return (eng.precision, eng._stamp, eng.vis.T * eng.vis.d, str(eng.device))

    def _ensure(self, eng):
        """(Re)allocates the buffers when the engine's staging changed (precision switch, frozen weights
        edited or reloaded, device move): everything cached before is invalid.  Returns True when the cache
        was (re)initialised, i.e. holds nothing."""
        stamp = self._stamp_of(eng)
        if self.x is None or self.stamp != stamp:
            width = stamp[2]
            self.x = torch.empty(self.capacity, width, device=eng.device)
            self.a = torch.empty(self.capacity, width, device=eng.device)
            self.present = set()
            self.stamp = stamp
            return True
        return False

    def all_present(self, ids, eng=None):
        """With `eng`: also validates that the entries were produced by the engine's CURRENT staging (and that
        the engine itself is staged for the current precision mode) - a stale cache answers False, never a hit."""
        if eng is not None:
            if (eng.device is None or eng.precision != _PRECISION or self.x is None
                    or self.stamp != self._stamp_of(eng)):
                return False
        return all(int(i) in self.present for i in ids)

    def lookup_device_ids(self, eng, ids_dev):
        """Hit path with the ids already on the device (the caller has checked `all_present(ids, eng)`): no host
        work, no host->device copy - what a captured CUDA graph of the cached step replays."""
        if self._ensure(eng):
            raise RuntimeError("TrunkCache: the engine was restaged after the cache was filled (precision switch, "
                               "frozen weight change or device move); the cached activations are invalid - "
                               "check all_present(ids, eng) before a device-id lookup")
        B, d = ids_dev.numel(), eng.vis.d
        x = torch.index_select(self.x, 0, ids_dev, out=eng._buf("v.x", (B, self.x.shape[1])))
        a = torch.index_select(self.a, 0, ids_dev, out=eng._buf("v.acache", (B, self.x.shape[1])))
        return {"cache": self, "ids": None, "hit": True, "x": x.view(B * eng.vis.T, d),
                "a": a.view(B * eng.vis.T, d)}

    def lookup(self, eng, ids):
        self._ensure(eng)
        ids = [int(i) for i in ids]
        if max(ids) >= self.capacity or min(ids) < 0:
            raise RuntimeError("TrunkCache: image id outside the cache capacity")
        ids_dev = torch.tensor(ids, dtype=torch.int64, device=eng.device)
        ctx = {"cache": self, "ids": (ids, ids_dev), "hit": all(i in self.present for i in ids)}
        if ctx["hit"]:
            B, d = len(ids), eng.vis.d
            ctx["x"] = torch.index_select(self.x, 0, ids_dev, out=eng._buf("v.x", (B, self.x.shape[1]))
                                          ).view(B * eng.vis.T, d)
            ctx["a"] = torch.index_select(self.a, 0, ids_dev, out=eng._buf("v.acache", (B, self.x.shape[1]))
                                          ).view(B * eng.vis.T, d)
        return ctx

    def store(self, ids, x, a_f32):
        host, dev = ids
        self.x.index_copy_(0, dev, x.view(len(host), -1))
        self.a.index_copy_(0, dev, a_f32.view(len(host), -1))
        self.present.update(host)


def get_engine(model) -> Engine:
    eng = model.__dict__.get("_hba_engine")
    if eng is None:
        eng = Engine(model)
        model.__dict__["_hba_engine"] = eng
    return eng


class _ClipForward(torch.autograd.Function):
    """preds = CLIP(image, tokens); differentiable w.r.t. the adapter `out_proj.weight` tensors."""

    @staticmethod
    def forward(ctx, engine, images, tokens, pos_embedding, keys, *tensors):
        n = len(keys)
        weights, biases = tensors[:n], tensors[n:]
        v_ad = {k[1]: (w, b) for k, w, b in zip(keys, weights, biases) if k[0] == "v"}
        t_ad = {k[1]: (w, b) for k, w, b in zip(keys, weights, biases) if k[0] == "t"}
        need_grad = any(ctx.needs_input_grad[5:5 + n])
        if any(ctx.needs_input_grad[5 + n:]):
            raise RuntimeError("libhba: adapter biases are frozen on this path (NEW:535-536)")
        if ctx.needs_input_grad[1]:
            raise RuntimeError("libhba: gradients w.r.t. the input images are not supported")
        pred, saved = engine.run_forward(images, tokens, pos_embedding, v_ad, t_ad, need_grad)
        # the loss becomes an OUTPUT of this node: keeping it in ctx.saved as well would close a reference cycle
        # (node -> saved -> tensor -> grad_fn = node) that only the garbage collector breaks, and the step's
        # autograd graph (with AccumulateGrad nodes bound to this step's stream) would survive into the next
        # CUDA-graph capture
        loss = saved.pop("loss")
        ctx.engine, ctx.saved, ctx.keys = engine, saved, keys
        ctx.set_materialize_grads(False)
        if loss is None:
            return pred
        return pred, loss

    @staticmethod
    def backward(ctx, d_pred, d_loss=None):
        if d_pred is None and d_loss is None:
            return (None,) * (5 + 2 * len(ctx.keys))
        grads = ctx.engine.run_backward(ctx.saved, d_pred, d_loss)
        out = []
        for i, k in enumerate(ctx.keys):
            g = grads.get(k)
            if ctx.needs_input_grad[5 + i] and g is None:
                raise RuntimeError(f"libhba: no gradient path staged for adapter {k}")
            out.append(g if ctx.needs_input_grad[5 + i] else None)
        return (None, None, None, None, None, *out, *([None] * len(ctx.keys)))


def clip_forward(model, image, text, pos_embedding=False):
    """Entry point used by the plug-in CLIP module's ``forward`` (src/models/CLIPs/clip_hba/clip.py)."""
    if not image.is_cuda:
        raise RuntimeError("libhba has no CPU path: move the model and the images to a CUDA device "
                           "(sm_100a)")
    eng = get_engine(model)
    keys, weights, biases = [], [], []
    for side, blocks in (("v", model.visual.transformer.resblocks), ("t", model.transformer.resblocks)):
        for i, blk in enumerate(blocks):
            op = blk.attn.out_proj
            if not isinstance(op, torch.nn.Linear):
                keys.append((side, i))
                weights.append(op.weight)   # DoRALayer.weight property: merged W [out, in]
                biases.append(op.bias)
    eng.loss_out = None
    if torch.is_grad_enabled() and any(w.requires_grad for w in weights):
        out = _ClipForward.apply(eng, image, text, pos_embedding, tuple(keys), *weights, *biases)
        if isinstance(out, tuple):
            out, eng.loss_out = out
        return out
    with torch.no_grad():
        v_ad = {k[1]: (w, b) for k, w, b in zip(keys, weights, biases) if k[0] == "v"}
        t_ad = {k[1]: (w, b) for k, w, b in zip(keys, weights, biases) if k[0] == "t"}
        pred, saved = eng.run_forward(image, text, pos_embedding, v_ad, t_ad, False)
        eng.loss_out = saved["loss"]
    return pred
