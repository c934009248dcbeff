"""fp64 references of the row-wise kernels (LayerNorm forward / backward / parameter gradients, column sums, token
assembly), a per-element error bound from an fp32 error analysis of the kernels' own arithmetic, the branch map of
their launchers, inputs that expose a wrong row statistic, and an fp32 emulation of the kernels for mutation checks.

References are computed in fp64 from the exact fp32 values handed to the kernel; `eps` is the fp32 value the kernel
receives.  LayerNorm uses the biased variance.

Error bound (u = 2^-24, g(k) = k u / (1 - k u); h = ceil(cols / 128) + 6)
  Every row statistic is a lane-partial sum - per lane (a + b) + (c + d) of each float4, the float4s of the lane in
  sequence - followed by 5 xor-shuffle levels: a summation tree of depth <= h, so |s_hat - s| <= g(h) sum |terms|.
  mean     mu_hat = fl(S / n) (bwd_fused: S * fl(1/n), one rounding more):  e_mu <= g(h + 2) A,  A = mean |x|.
  variance sum (x - mu_hat)^2 = n (var + e_mu^2) exactly (the cross term vanishes); each centred value is rounded once,
           squared with one rounding, summed with depth h and divided: v_hat = (var + e_mu^2)(1 + t), |t| <= g(h + 4);
           + eps rounds once more.  rsqrtf is good to 2 ulp (2^-22 relative), so r_hat = r (1 + rho),
           rho <= q / (2 (1 - q)) + 2^-22,  q = (g(h + 4) (var + e_mu^2) + e_mu^2) / (var + eps) + u.
           The e_mu terms make the bound absolute per row: in a constant row the reference y is exactly beta while
           the kernel's mean is off by up to e_mu, and (x - mu_hat) r gamma is then e_mu r |gamma|, not 0.
  xhat     xhat_hat = fl(fl(x - mu_hat) r_hat):  E_xhat <= r e_mu (1 + rho + 2u) + |xhat| ((1 + rho)(1 + u)^2 - 1).
  forward  y = fl(fl(xhat_hat gamma) + beta) (an FMA rounds less):  E_y <= (1 + u) |gamma| E_xhat' + u |y|, where
           E_xhat' adds one rounding for the product.
  backward g = fl(dy gamma); s1 = fl(sum g) / n, s2 = fl(sum fl(g xhat_hat)) / n (depth h, + 1 for bwd_fused's 1/n);
           z = fl(fl(g - s1) - fl(xhat_hat s2)); dx = fl(r_hat z):
           e_s1 <= g(h + 3) mean|g|,  e_s2 <= mean(|g| E_xhat) + g(h + 4) mean(|g| (|xhat| + E_xhat)),
           e_z  <= u |g| + e_s1 + E_xhat |s2| + (|xhat| + E_xhat) e_s2 + 3u (|g| + |s1| + (|xhat| + E_xhat) |s2|),
           E_dx <= r (1 + rho)(1 + u) e_z + (rho + 2u) r |z|.  With dy in the null space of the Jacobian z is a small
           difference of large terms, and the bound is set by |g|, |s1| and |xhat s2|, not by |dx|.
  accumulate  one more rounding: + u (|ref| + E).
  column sums (colsum, param_grad): a thread adds every 8th row of a chunk of per = ceil(rows / 128) rows, the 8 row
           phases are added in turn, then the 128 chunks: depth D = ceil(per / 8) + 8 + 128 (+ 1 with accumulate),
           error g(D) sum |terms| plus the per-term errors (dy xhat_hat: |dy| (E_xhat + 2u (|xhat| + E_xhat))).
           bwd_fused: a warp adds its rows (cyclic over 8 * blocks warps), the 8 warps of a block are added in turn,
           then the blocks in 4 interleaved partial sums combined pairwise: D = ceil(rows / (8 blocks)) + 8 +
           ceil(blocks / 4) + 2.
  output   one rounding of the stored type: 0 for f32, 2^-8 for a bf16 hi part, 2^-16 for hi + lo.
The bound is an a-priori worst case.  Its summation terms are far from attained (random-sign rounding errors grow
like sqrt(depth)), but a single final rounding - y = ... + beta with |beta| >> |gamma xhat|, an accumulated value, a
bf16 hi part - is bounded by its exact worst case (half an ulp), which a value just above a power of two attains: on
such paths the worst observed |out - ref| / bound sits just below 1, as it must.  Sensitivity comes from the inputs
(`ln_rows`, `ln_params`, `bwd_dy`).
"""
from __future__ import annotations

import math

import torch

U32 = 2.0 ** -24
RSQRT = 2.0 ** -22                 # 2 ulp of rsqrtf, relative
NUM_SMS = 148                      # B200
LNS_ROWS = 24                      # rowwise.cu kLnsRows: consumer warps = rows per stage
LNS_MAX_STAGES = 8
CS_CHUNKS = 128                    # vit_extra.cu kCsChunks
FUSED_COLS = (128, 256, 512, 768, 1024)
OUT_ROUNDING = {"f32": 0.0, "bf16": 2.0 ** -8, "hilo": 2.0 ** -16}
EPS_CLIP, EPS_TIMM = 1e-5, 1e-6


def gam(k):
    return k * U32 / (1 - k * U32)


def f32(v):
    """The fp32 value a float argument becomes at the C-ABI."""
    return float(torch.tensor(v, dtype=torch.float32))


def depth(cols):
    return -(-cols // 128) + 6


# ---------------------------------------------------------------------------------------- references (fp64)
def ln_stats(x, eps):
    """x [R, n] (fp32 values) -> fp64 dict: mean, var (biased), rstd = 1 / sqrt(var + fp32(eps)), xhat, A = mean |x|."""
    xd = x.double()
    mu = xd.mean(1, keepdim=True)
    var = ((xd - mu) ** 2).mean(1, keepdim=True)
    r = 1.0 / torch.sqrt(var + f32(eps))
    return {"x": xd, "mean": mu, "var": var, "rstd": r, "xhat": (xd - mu) * r, "A": xd.abs().mean(1, keepdim=True),
            "eps": f32(eps), "cols": x.shape[1]}


def ln_fwd_ref(x, gamma, beta, eps):
    st = ln_stats(x, eps)
    st["gamma"], st["beta"] = gamma.double(), beta.double()
    st["y"] = st["xhat"] * st["gamma"] + st["beta"]
    return st


def ln_bwd_ref(dy, x, gamma, eps, prev=None):
    """dx = rstd (g - mean g - xhat mean(g xhat)), g = dy gamma (+ prev with accumulate)."""
    st = ln_stats(x, eps)
    g = dy.double() * gamma.double()
    s1 = g.mean(1, keepdim=True)
    s2 = (g * st["xhat"]).mean(1, keepdim=True)
    z = g - s1 - st["xhat"] * s2
    st.update(dy=dy.double(), g=g, s1=s1, s2=s2, z=z, dx=st["rstd"] * z)
    st["prev"] = prev.double() if prev is not None else None
    if prev is not None:
        st["dx"] = st["dx"] + st["prev"]
    return st


def param_grad_ref(dy, x, eps):
    """(dgamma, dbeta) = (sum_r dy xhat, sum_r dy) and the row statistics."""
    st = ln_stats(x, eps)
    d = dy.double()
    st.update(dy=d, dgamma=(d * st["xhat"]).sum(0), dbeta=d.sum(0))
    return st


def colsum_ref(x):
    return x.double().sum(0)


def assemble_x(conv, cls, pos, B, n_patches):
    """The fp32 token rows the kernel normalises: fl(cls + pos[0]), fl(conv[b, p] + pos[1 + p]) (one IEEE add)."""
    w = conv.shape[1]
    c = conv.reshape(B, n_patches, w)
    return (torch.cat([cls.reshape(1, 1, w).expand(B, 1, w), c], 1) + pos[:n_patches + 1]).reshape(-1, w)


# ---------------------------------------------------------------------------------------- error bound
def stat_errors(st, fused=False):
    """e_mu, rho (per row) and E_xhat (per element) of the kernel's statistics."""
    h = depth(st["cols"]) + (1 if fused else 0)
    e_mu = gam(h + 2) * st["A"]
    var = st["var"]
    q = (gam(h + 4) * (var + e_mu ** 2) + e_mu ** 2) / (var + st["eps"]) + U32
    rho = q / (2 * (1 - q)) + RSQRT * (1 + q)
    ex = st["rstd"] * e_mu * (1 + rho + 2 * U32) + st["xhat"].abs() * ((1 + rho) * (1 + U32) ** 2 - 1)
    return e_mu, rho, ex


def _stored(e, ref, out):
    return e + OUT_ROUNDING[out] * (ref.abs() + e)


def ln_fwd_bound(st, out="f32"):
    _, _, ex = stat_errors(st)
    ga = st["gamma"].abs()
    e = (1 + U32) * ga * (ex + U32 * (st["xhat"].abs() + ex)) + U32 * st["y"].abs()
    return _stored(e, st["y"], out)


def ln_bwd_bound(st, fused=False, out="f32"):
    h = depth(st["cols"]) + (1 if fused else 0)
    _, rho, ex = stat_errors(st, fused)
    g, s1, s2, xa, r = st["g"].abs(), st["s1"].abs(), st["s2"].abs(), st["xhat"].abs(), st["rstd"]
    e_s1 = gam(h + 3) * g.mean(1, keepdim=True)
    e_s2 = (g * ex).mean(1, keepdim=True) + gam(h + 4) * (g * (xa + ex)).mean(1, keepdim=True)
    e_z = U32 * g + e_s1 + ex * s2 + (xa + ex) * e_s2 + 3 * U32 * (g + s1 + (xa + ex) * s2)
    e = r * (1 + rho) * (1 + U32) * e_z + (rho + 2 * U32) * r * st["z"].abs()
    if st["prev"] is not None:
        e = e + U32 * (st["dx"].abs() + e)
    return _stored(e, st["dx"], out)


def colsum_depth(rows):
    per = -(-rows // CS_CHUNKS)
    return -(-per // 8) + 8 + CS_CHUNKS


def fused_depth(rows, num_sms=NUM_SMS):
    blocks = bwd_fused_branches(rows, 128, num_sms)["blocks"]
    return -(-rows // (8 * blocks)) + 8 + -(-blocks // 4) + 2


def colsum_bound(x, prev=None, D=None):
    """Column sums of x [rows, cols] (f32 or bf16 values, or the kernel's own dx for bwd_fused: pass D)."""
    D = colsum_depth(x.shape[0]) if D is None else D
    ref = colsum_ref(x)
    e = gam(D) * x.double().abs().sum(0)
    if prev is not None:
        ref = ref + prev.double()
        e = e + U32 * (ref.abs() + e)
    return ref, e


def param_grad_bound(st, prev=None, D=None, fused=False):
    """(dgamma | dbeta reference, bound) for param_grad (column-sum depth) or bwd_fused (D = fused_depth)."""
    rows = st["dy"].shape[0]
    D = colsum_depth(rows) if D is None else D
    _, _, ex = stat_errors(st, fused)
    d, xa = st["dy"].abs(), st["xhat"].abs()
    eg = (d * (ex + 2 * U32 * (xa + ex))).sum(0) + gam(D) * (d * (xa + ex)).sum(0)
    eb = gam(D) * d.sum(0)
    ref = torch.cat([st["dgamma"], st["dbeta"]])
    e = torch.cat([eg, eb])
    if prev is not None:
        ref = ref + prev.double()
        e = e + U32 * (ref.abs() + e)
    return ref, e


# ---------------------------------------------------------------------------------------- branch map
def ln_fwd_stages(cols):
    """rowwise.cu:460-461: ring stages of 24 rows that fit 220 KB next to gamma and beta."""
    return min(LNS_MAX_STAGES, (220 * 1024 - 2 * cols * 4 - 256) // (LNS_ROWS * cols * 4))


def ln_fwd_branches(rows, cols, num_sms=NUM_SMS):
    """What hba_layernorm_fwd does (rowwise.cu:449-476): the per-row kernel below 1024 rows (8 rows per block),
    otherwise the streaming kernel: persistent CTAs (148, or ceil(rows / 24) below 148 x 24 = 3552 rows), CTA b owning
    rows [rows b / grid, rows (b + 1) / grid) (:156), pulled through the ring in iterations of 24 rows (:157); the
    producer waits on the empty barrier from iteration `stages` on (:175), i.e. the ring wraps; a last iteration of
    fewer than 24 rows leaves consumer warps idle."""
    if rows < 1024:
        return {"form": "per_row", "blocks": -(-rows // 8)}
    stages = ln_fwd_stages(cols)
    grid = num_sms if num_sms * LNS_ROWS <= rows else -(-rows // LNS_ROWS)
    per = [rows * (b + 1) // grid - rows * b // grid for b in range(grid)]
    iters = [-(-n // LNS_ROWS) for n in per]
    return {"form": "stream", "stages": stages, "grid": grid, "rows_min": min(per), "rows_max": max(per),
            "iters_min": min(iters), "iters_max": max(iters), "wraps": (max(iters) - 1) // stages,
            "partial_last": any(n % LNS_ROWS for n in per), "per_cta": per}


def bwd_fused_branches(rows, cols, num_sms=NUM_SMS):
    """vit_extra.cu:482-497: NVEC = cols / 128, blocks = min(2 * #SM, ceil(rows / 8)), rows cyclic over the warps."""
    blocks = min(2 * num_sms, -(-rows // 8))
    return {"nvec": cols // 128, "blocks": blocks, "rows_per_warp_max": -(-rows // (8 * blocks)),
            "rows_per_warp_min": rows // (8 * blocks)}


def colsum_branches(rows, cols):
    """vit_extra.cu:32-33, 54-55: chunk k owns rows [k per, min((k + 1) per, rows)), per = ceil(rows / 128); chunks past
    the last row are empty; column blocks of 32, the last one partial when cols % 32 != 0."""
    per = -(-rows // CS_CHUNKS)
    used = -(-rows // per)
    return {"per": per, "empty_chunks": CS_CHUNKS - used, "col_blocks": -(-cols // 32), "partial_col_block": cols % 32 != 0}


def wrap_rows(cols, wraps=2, extra=5, num_sms=NUM_SMS):
    """Rows that give every CTA of the streaming form (wraps x stages + 1) full iterations plus a partial one of
    `extra` rows: the ring wraps `wraps` times and the last stage leaves 24 - extra consumer warps idle."""
    return num_sms * (LNS_ROWS * (wraps * ln_fwd_stages(cols) + 1) + extra)


# ---------------------------------------------------------------------------------------- inputs
ROW_KINDS = ("normal", "offset", "tiny_var", "constant", "outlier", "zero")


def ln_rows(rows, cols, seed=0, eps=EPS_CLIP):
    """fp32 [rows, cols]; row r has kind ROW_KINDS[r % 6] (rotated by seed):
      normal    mu + sigma z, sigma = 2^U[-3, 3], mu = sigma N(0, 1)
      offset    mu + sigma z with |mu| / sigma = 2^U[4, 10] (a wrong or short mean sum moves every element)
      tiny_var  sigma^2 = eps 2^-12 around a mean of order one: var << eps
      constant  every element equal (the reference is exactly beta)
      outlier   a normal row with one column at 64 sigma (the CLIP residual stream has such features)
      zero      all zeros"""
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(rows, cols, generator=g, dtype=torch.float64)
    sig = torch.exp2(torch.randint(-3, 4, (rows, 1), generator=g).double())
    mu = torch.randn(rows, 1, generator=g, dtype=torch.float64) * sig
    kind = (torch.arange(rows) + seed) % len(ROW_KINDS)
    x = mu + sig * z
    off = kind == 1
    sgn = torch.where(torch.rand(rows, 1, generator=g) < 0.5, -1.0, 1.0).double()
    ratio = torch.exp2(4 + 6 * torch.rand(rows, 1, generator=g, dtype=torch.float64))
    x[off] = (sgn * ratio * sig + sig * z)[off]
    tiny = kind == 2
    x[tiny] = (mu / sig + math.sqrt(eps) * 2.0 ** -6 * z)[tiny]
    const = kind == 3
    x[const] = (mu * 3).expand(rows, cols)[const]
    out = kind == 4
    col = torch.randint(0, cols, (rows,), generator=g)
    spike = torch.zeros(rows, cols, dtype=torch.float64)
    spike[torch.arange(rows), col] = 64.0
    x[out] = (x + spike * sig)[out]
    x[kind == 5] = 0.0
    return x.float()


def strided(x, row_step, seed=0):
    """A [rows * row_step, cols] source whose rows r * row_step are x's rows (every row kind stays present) and
    whose rows in between are other normal values."""
    rows, cols = x.shape
    full = torch.randn(rows * row_step, cols, generator=torch.Generator().manual_seed(seed + 55)) * 3
    full[::row_step] = x
    return full


def ln_params(cols, seed=0, zeros=True):
    """gamma |N(0, 1)| + 0.05 with alternating signs and (zeros=True) every 7th entry 0; beta 16 N(0, 1): large next
    to gamma xhat.  The backward cases take zeros=False: where gamma is 0, g = dy gamma cannot follow the null space."""
    g = torch.Generator().manual_seed(seed + 101)
    gamma = torch.randn(cols, generator=g).abs() + 0.05
    gamma = gamma * torch.where(torch.arange(cols) % 2 == 0, 1.0, -1.0)
    if zeros:
        gamma[::7] = 0.0
    beta = 16 * torch.randn(cols, generator=g)
    return gamma, beta


def bwd_dy(x, gamma, eps, seed=0):
    """dy [rows, cols]: row kinds rotate over
      null     dy_c = (a + b xhat_c) / gamma_c + 2^-10 N(0, 1): g = dy gamma lies in the null space of the LayerNorm
               Jacobian up to the noise, so dx is a small difference of large terms (N(0, 1) where gamma_c = 0)
      column   all of dy on one column
      normal   N(0, 1) times a row scale 2^U[-4, 4]"""
    rows, cols = x.shape
    g = torch.Generator().manual_seed(seed + 7)
    xhat = ln_stats(x, eps)["xhat"]
    gd = gamma.double()
    noise = torch.randn(rows, cols, generator=g, dtype=torch.float64)
    a = 4 * torch.randn(rows, 1, generator=g, dtype=torch.float64)
    b = 4 * torch.randn(rows, 1, generator=g, dtype=torch.float64)
    safe = torch.where(gd == 0, 1.0, gd)
    null = torch.where(gd == 0, noise, (a + b * xhat) / safe + 2.0 ** -10 * noise)
    col = torch.zeros(rows, cols, dtype=torch.float64)
    col[torch.arange(rows), torch.randint(0, cols, (rows,), generator=g)] = 3 * a[:, 0]
    normal = noise * torch.exp2(torch.randint(-4, 5, (rows, 1), generator=g).double())
    kind = (torch.arange(rows) + seed) % 3
    dy = torch.where((kind == 0)[:, None], null, torch.where((kind == 1)[:, None], col, normal))
    return dy.float()


# ---------------------------------------------------------------------------------------- fp32 emulation of the kernels
def _lane_sum(t4, skip_chunk=False):
    """The kernels' row sum of float4 terms t4 [R, nvec, 32, 4] (fp32): per lane (a + b) + (c + d), the lane's float4s
    in sequence, then the xor-shuffle tree.  skip_chunk drops lane 31's last float4 (a mutant)."""
    p = (t4[..., 0] + t4[..., 1]) + (t4[..., 2] + t4[..., 3])
    if skip_chunk:
        p = p.clone()
        p[:, -1, 31] = 0
    s = p[:, 0]
    for i in range(1, p.shape[1]):
        s = s + p[:, i]
    lanes = torch.arange(32)
    for o in (16, 8, 4, 2, 1):
        s = s + s[:, lanes ^ o]
    return s[:, :1]


def _as4(v):
    R, n = v.shape
    return v.reshape(R, n // 128, 32, 4)


def _stats32(x, eps, mutant=None):
    n = x.shape[1]
    skip = mutant == "skip_chunk"
    mean = _lane_sum(_as4(x), skip) / n
    d = x - mean
    var = _lane_sum(_as4(d * d), skip) / (n - 1 if mutant == "unbiased" else n)
    if mutant == "eps_outside":
        rstd = (1.0 / (torch.sqrt(var.double()) + f32(eps))).float()
    else:
        rstd = (1.0 / torch.sqrt((var + torch.tensor(eps, dtype=torch.float32)).double())).float()
    return d, rstd


def emulate_ln_fwd(x, gamma, beta, eps, mutant=None):
    """layernorm_fwd_kernel in fp32 on the CPU (same summation order, correctly rounded rsqrt).  Mutants: "unbiased",
    "eps_outside", "skip_chunk", "drop_last_stage" (the streaming form forgets the partial last stage of each CTA:
    those rows keep the output's previous contents, zeros here)."""
    x = x.float()
    d, rstd = _stats32(x, eps, mutant)
    y = (d * rstd) * gamma + beta
    if mutant == "drop_last_stage":
        br = ln_fwd_branches(x.shape[0], x.shape[1])
        start = 0
        for n in br["per_cta"]:
            if n % LNS_ROWS:
                y[start + n - n % LNS_ROWS:start + n] = 0
            start += n
    return y


def emulate_ln_bwd(dy_buf, x, gamma, eps, prev=None, row_step=1, mutant=None):
    """layernorm_bwd_kernel in fp32: x rows are taken at r * row_step (x is the strided source), dy and dx rows at r.
    Mutants: "dy_row_step" (dy read at r * row_step too), "wrong_row" (accumulation reads the previous dx of row
    r + 1), "unbiased", "eps_outside", "skip_chunk"."""
    rows = x.shape[0]
    dy = dy_buf[::row_step][:rows] if mutant == "dy_row_step" else dy_buf[:rows]
    d, rstd = _stats32(x.float(), eps, mutant)
    xh = d * rstd
    g = dy * gamma
    n = x.shape[1]
    s1 = _lane_sum(_as4(g)) / n
    s2 = _lane_sum(_as4(g * xh)) / n
    o = rstd * ((g - s1) - xh * s2)
    if prev is not None:
        o = o + (torch.roll(prev, -1, 0) if mutant == "wrong_row" else prev)
    return o
