"""RSA evaluation on the GPU (replaces the NumPy/SciPy tail of the reference's behavioral_RSA,
NEW:625-652, and of compute_rsa_score, MEAS:298-355):

    model_rdm = 1 - corrcoef(E)  (float64, diag 0)  ->  upper triangle (k=1, row-major)
    rho = Pearson(rank_avg(reference_tri), rank_avg(model_tri))     (= scipy.stats.spearmanr)

Only the Student-t survival function for the p-value is evaluated on the host (one scalar).

Resampling statistics (RSAEvaluator.permutation_test / .bootstrap) resample stimuli, the unit the RDM entries depend
on: a Mantel permutation test for the p-value and the stimulus bootstrap of Nili et al. 2014 for confidence intervals.
Replicates are drawn on the host (numpy.random.default_rng(seed)) and evaluated by hba_rsa_perm_null /
hba_rsa_bootstrap, each RDM sorted once (hba_rank_order_f64).

RSAEvaluator.kendall_tau compares the two RDMs with Kendall's tau-a and tau-b instead of rho (hba_kendall_tau_f64,
against the same cached sorted order of the reference).
"""
from __future__ import annotations

import numpy as np
import torch

from . import ops

# device memory a resampling call may hold at once (workspace, replicate uploads, outputs); replicates go to the device
# in chunks that fit it
STATS_CHUNK_BYTES = 1 << 30


class RSAEvaluator:
    """Holds the ranked reference RDM and the workspaces for repeated evaluations of N x D
    embeddings against one reference RDM."""

    def __init__(self, reference_rdm, device="cuda"):
        ref = np.asarray(reference_rdm, dtype=np.float64)
        if ref.ndim != 2 or ref.shape[0] != ref.shape[1]:
            raise ValueError("reference_rdm must be a square matrix")
        self.N = ref.shape[0]
        self.P = self.N * (self.N - 1) // 2
        self.device = torch.device(device)
        iu = np.triu_indices(self.N, k=1)
        ref_tri = torch.from_numpy(np.ascontiguousarray(ref[iu])).to(self.device)
        self.rank_ws = torch.empty(max(ops.rank_workspace_bytes(self.P), 256), dtype=torch.uint8,
                                   device=self.device)
        self.ref_ranks = torch.empty(self.P, dtype=torch.float64, device=self.device)
        ops.rank_avg_f64(ref_tri, self.ref_ranks, self.rank_ws)
        self.ref_tri = ref_tri
        self._ref_order = None
        self._kendall = None     # (workspace, counts [4] int64, tau [2] f64) of kendall_tau, allocated on first use
        self.tri = torch.empty(self.P, dtype=torch.float64, device=self.device)
        self.ranks = torch.empty(self.P, dtype=torch.float64, device=self.device)
        self.rdm = torch.empty(self.N, self.N, dtype=torch.float64, device=self.device)
        self.pearson_ws = torch.empty(5 * 1024, dtype=torch.float64, device=self.device)
        self.rho = torch.empty(1, dtype=torch.float64, device=self.device)

    def rho_device(self, emb, want_rdm=True):
        """Launches the whole chain on the current stream; returns the device scalar rho."""
        if emb.shape[0] != self.N:
            raise ValueError(f"expected {self.N} embeddings, got {emb.shape[0]}")
        emb = emb.detach().to(self.device, torch.float32).contiguous()
        if self.P > 2048:
            # RSA at scale: one fused chain (keys straight from the RDM kernel, ranks consumed in sorted order)
            ops.rdm_spearman(emb, self.ref_ranks, self.rho, self.rank_ws, rdm=self.rdm if want_rdm else None)
            return self.rho
        ops.rdm_f64(emb, self.rdm if want_rdm else None, self.tri)
        ops.rank_avg_f64(self.tri, self.ranks, self.rank_ws)
        ops.pearson_f64(self.ref_ranks, self.ranks, self.rho, self.pearson_ws)
        return self.rho

    def __call__(self, emb, want_rdm=True):
        """-> (rho, p_value, model_rdm ndarray | None), like behavioral_RSA's return (NEW:654)."""
        with torch.cuda.device(self.device):
            rho = float(self.rho_device(emb, want_rdm).cpu())
        rdm = self.rdm.cpu().numpy() if want_rdm else None
        return rho, spearman_pvalue(rho, self.P), rdm

    # ------------------------------------------------------------------ resampling statistics
    def _observed(self, emb):
        with torch.cuda.device(self.device):
            return float(self.rho_device(emb, want_rdm=False).cpu())

    def _model_arrays(self, emb):
        """(upper triangle [P] f64, its stable sorted order [P] int32, its average ranks [P] f64) of emb's RDM."""
        emb = emb.detach().to(self.device, torch.float32).contiguous()
        tri = torch.empty(self.P, dtype=torch.float64, device=self.device)
        order = torch.empty(self.P, dtype=torch.int32, device=self.device)
        ranks = torch.empty(self.P, dtype=torch.float64, device=self.device)
        ops.rdm_f64(emb, None, tri)
        ops.rank_order_f64(tri, order, ranks, self.rank_ws)
        return tri, order, ranks

    def _reference_order(self):
        """The stable sorted order [P] int32 of the reference triangle (hba_rank_order_f64), computed once."""
        if self._ref_order is None:
            self._ref_order = torch.empty(self.P, dtype=torch.int32, device=self.device)
            ranks = torch.empty(self.P, dtype=torch.float64, device=self.device)
            ops.rank_order_f64(self.ref_tri, self._ref_order, ranks, self.rank_ws)
        return self._ref_order

    def _chunk(self, n, bytes_of, per_replicate_host):
        """Replicates per device call so that workspace + uploads + outputs stay within STATS_CHUNK_BYTES."""
        one, two = bytes_of(1), bytes_of(2)
        per = (two - one) + per_replicate_host
        return int(max(1, min(n, (STATS_CHUNK_BYTES - (one - (two - one))) // per)))

    def permutation_test(self, emb, n_perm=10000, seed=0):
        """Mantel test of the Spearman rho of emb's RDM against the reference: the stimuli of the model RDM are
        relabelled by n_perm random permutations.  -> (rho, p_perm, null [n_perm] f64) with the one-sided
        p_perm = (1 + #{null >= rho}) / (1 + n_perm).  A NaN rho gives p_perm = NaN and an all-NaN null.

        Draw order: rng = numpy.random.default_rng(seed); permutation p is rng.permutation(N), p = 0, 1, ... - so every
        checkpoint evaluated with the same seed sees the same permutations."""
        if n_perm < 1:
            raise ValueError("n_perm must be >= 1")
        rho = self._observed(emb)
        null = np.full(n_perm, np.nan)
        if rho != rho:
            return rho, float("nan"), null
        rng = np.random.default_rng(seed)
        with torch.cuda.device(self.device):
            _, _, ranks = self._model_arrays(emb)
            chunk = self._chunk(n_perm, lambda k: ops.rsa_perm_workspace_bytes(self.N, k), 4 * self.N + 8)
            ws = torch.empty(ops.rsa_perm_workspace_bytes(self.N, chunk), dtype=torch.uint8, device=self.device)
            for s in range(0, n_perm, chunk):
                k = min(chunk, n_perm - s)
                perms = np.stack([rng.permutation(self.N) for _ in range(k)]).astype(np.int32)
                check_permutations(perms, self.N)
                out = torch.full((k,), float("nan"), dtype=torch.float64, device=self.device)
                ops.rsa_perm_null(self.ref_ranks, ranks, torch.from_numpy(perms).to(self.device), out, ws)
                null[s:s + k] = out.cpu().numpy()
        return rho, permutation_pvalue(rho, null), null

    def bootstrap(self, emb, n_boot=1000, seed=0, alpha=0.05, paired_with=None):
        """Stimulus bootstrap (Nili et al. 2014) of the Spearman rho of emb's RDM against the reference: each replicate
        draws N stimuli with replacement; a pair {i, j} of distinct stimuli then enters with multiplicity c_i c_j and
        pairs of a stimulus with itself are dropped.  With paired_with (embeddings of another model on the same
        images) every replicate is rho(emb) - rho(paired_with) on the identical resample.
        -> ((lo, hi), replicates [n_boot] f64, n_valid): the percentile interval np.quantile(valid, [alpha/2,
        1 - alpha/2]) over the valid replicates.  A replicate whose resampled triangle is constant or holds a NaN (so
        one with fewer than 3 distinct stimuli) is NaN and not valid.  A NaN observed rho (difference) gives a NaN
        interval, all-NaN replicates and n_valid = 0.

        Draw order: rng = numpy.random.default_rng(seed); replicate b takes idx = rng.integers(0, N, size=N) and
        counts c = numpy.bincount(idx, minlength=N), b = 0, 1, ... - so every checkpoint evaluated with the same seed
        sees the same resamples."""
        if n_boot < 1:
            raise ValueError("n_boot must be >= 1")
        if not 0.0 < alpha < 1.0:
            raise ValueError("alpha must be in (0, 1)")
        obs = self._observed(emb)
        if paired_with is not None:
            obs -= self._observed(paired_with)
        reps = np.full(n_boot, np.nan)
        if obs != obs:
            return (float("nan"), float("nan")), reps, 0
        rng = np.random.default_rng(seed)
        with torch.cuda.device(self.device):
            ref_order = self._reference_order()
            tri_a, order_a, _ = self._model_arrays(emb)
            tri_b = order_b = None
            if paired_with is not None:
                tri_b, order_b, _ = self._model_arrays(paired_with)
            chunk = self._chunk(n_boot, lambda k: ops.rsa_boot_workspace_bytes(self.N, k), 4 * self.N + 16)
            ws = torch.empty(ops.rsa_boot_workspace_bytes(self.N, chunk), dtype=torch.uint8, device=self.device)
            for s in range(0, n_boot, chunk):
                k = min(chunk, n_boot - s)
                counts = np.stack([np.bincount(rng.integers(0, self.N, size=self.N), minlength=self.N)
                                   for _ in range(k)]).astype(np.int32)
                counts_dev = torch.from_numpy(counts).to(self.device)
                out_a = torch.full((k,), float("nan"), dtype=torch.float64, device=self.device)
                out_b = None if tri_b is None else torch.full((k,), float("nan"), dtype=torch.float64,
                                                              device=self.device)
                ops.rsa_bootstrap(self.ref_tri, ref_order, tri_a, order_a, counts_dev, out_a, ws,
                                  tri_b=tri_b, order_b=order_b, rho_b=out_b)
                r = out_a.cpu().numpy()
                if out_b is not None:
                    r = r - out_b.cpu().numpy()
                reps[s:s + k] = r
        return percentile_interval(reps, alpha), reps, int(np.isfinite(reps).sum())

    # ------------------------------------------------------------------ Kendall's tau
    def kendall_tau(self, emb):
        """Kendall's tau of emb's RDM (x) against the reference (y) over the P upper-triangle pairs, from exact pair
        counts on the device (hba_kendall_tau_f64) -> (tau_a, tau_b).  tau_b equals scipy.stats.kendalltau; tau_a =
        (concordant - discordant) / (P (P - 1) / 2) does not favour model RDMs that predict tied dissimilarities, which
        is why Nili et al. 2014 recommend it whenever either RDM has ties (e.g. a categorical reference).  NaN when an
        RDM entry is NaN or when either triangle is constant."""
        if emb.shape[0] != self.N:
            raise ValueError(f"expected {self.N} embeddings, got {emb.shape[0]}")
        with torch.cuda.device(self.device):
            emb = emb.detach().to(self.device, torch.float32).contiguous()
            if self._kendall is None:
                ws = torch.empty(ops.kendall_workspace_bytes(self.P), dtype=torch.uint8, device=self.device)
                self._kendall = (ws, torch.empty(4, dtype=torch.int64, device=self.device),
                                 torch.empty(2, dtype=torch.float64, device=self.device))
            ws, counts, tau = self._kendall
            ops.rdm_f64(emb, None, self.tri)
            ops.kendall_tau_f64(self.tri, self.ref_tri, self._reference_order(), counts, tau, ws)
            tau_a, tau_b = tau.cpu().tolist()
        return tau_a, tau_b


def spearman_pvalue(rho, n):
    """Two-sided p-value of scipy.stats.spearmanr: t = r sqrt(dof / ((r+1)(1-r))), dof = n-2."""
    from scipy import special
    dof = n - 2
    if dof <= 0 or rho != rho:   # scipy returns (nan, nan) for constant / NaN input
        return float("nan")
    denom = (rho + 1.0) * (1.0 - rho)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = rho * np.sqrt(max(dof / denom, 0.0)) if denom > 0 else np.inf * np.sign(rho)
    return float(2.0 * special.stdtr(dof, -abs(t)))


def check_permutations(perms, N):
    """Raises ValueError unless every row of perms [n, N] is a permutation of 0..N-1."""
    perms = np.asarray(perms)
    if perms.ndim != 2 or perms.shape[1] != N or not (np.sort(perms, axis=1) == np.arange(N)).all():
        raise ValueError(f"every row must be a permutation of 0..{N - 1}")


def permutation_pvalue(rho, null):
    """One-sided Mantel p-value (1 + #{null >= rho}) / (1 + len(null)); NaN for a NaN rho."""
    if rho != rho:
        return float("nan")
    null = np.asarray(null, dtype=np.float64)
    return float((1 + np.count_nonzero(null >= rho)) / (1 + len(null)))


def percentile_interval(replicates, alpha=0.05):
    """(lo, hi) = np.quantile(valid, [alpha/2, 1 - alpha/2]) over the finite replicates; NaN when there are none."""
    r = np.asarray(replicates, dtype=np.float64)
    valid = r[np.isfinite(r)]
    if valid.size == 0:
        return float("nan"), float("nan")
    lo, hi = np.quantile(valid, [alpha / 2, 1 - alpha / 2])
    return float(lo), float(hi)


def rsa_from_embeddings(emb, reference_rdm):
    return RSAEvaluator(reference_rdm, emb.device)(emb)
