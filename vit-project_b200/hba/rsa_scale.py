"""RSA evaluation at scale (BASELINE.json configs[4]): for every DoRA checkpoint `epoch{N}_dora_params.pth` of a
baseline run or of the sweep conditions, the 66-D CLIP-HBA embeddings of ALL images of the set (1,854 THINGS
images = 1,806 training / test images + the 48 RSA images in the reference's files), their RDM and Spearman's rho
against a reference RDM - NEW:605-654 applied to N = 1,854 (P = 1,717,731 pairs) per checkpoint.

What is cheap here and expensive in the reference:
  * the embeddings of a checkpoint only need the LIVE sub-graph (block L-2 from its attention output on, the CLS row
    of block L-1, the text tail): the frozen trunk of every image comes from the HBM trunk cache (filled once per
    process, hba.engine.TrunkCache) and the forward batches replay as CUDA graphs
    (functions._pipeline_core._CachedForwardGraphs);
  * the tail (RDM in float64, average-tie ranking, Pearson on ranks) is hba_rdm_spearman: 11 launches, no host
    round trip (the reference: numpy.corrcoef + scipy.stats.spearmanr on the host, ~1.2 s per checkpoint at N = 1,854).
Checkpoints are independent (SURVEY 8e): rank r evaluates files r, r + W, ... ; the only communication is the
gather of the result rows on rank 0.
"""
from __future__ import annotations

import glob
import os
import re
import time

import numpy as np
import torch

RESULT_COLUMNS = ("checkpoint", "run", "epoch", "behavioral_rsa_rho", "behavioral_rsa_p_value")
# written only when asked for (n_perm > 0 / n_boot > 0): Mantel p-value, stimulus-bootstrap 95 % interval of rho
PERMUTATION_COLUMNS = ("behavioral_rsa_p_perm",)
BOOTSTRAP_COLUMNS = ("behavioral_rsa_ci_low", "behavioral_rsa_ci_high", "behavioral_rsa_boot_valid")
# written only with kendall=True: Kendall's tau-a and tau-b of the model RDM against the reference (RSAEvaluator.kendall_tau)
KENDALL_COLUMNS = ("behavioral_rsa_tau_a", "behavioral_rsa_tau_b")
_EPOCH = re.compile(r"epoch(\d+)_dora_params\.pth$")


def find_dora_checkpoints(root):
    """Every `epoch{N}_dora_params.pth` under `root` (a baseline run's dora directory, a sweep's output tree of
    SWEEP:198-207 / LEN:128-137, or both), sorted by (directory, epoch)."""
    files = [f for f in glob.glob(os.path.join(root, "**", "epoch*_dora_params.pth"), recursive=True)
             if _EPOCH.search(f)]
    return sorted(files, key=lambda f: (os.path.dirname(f), int(_EPOCH.search(f).group(1))))


def reference_rdm_from_targets(targets):
    """1 - corrcoef of the behavioural embedding itself (the SPoSE 66-D targets of the same images): the
    reference RDM of the full image set, as `RDM48_triplet` is for the 48-image subset (NEW:636-640)."""
    t = np.asarray(targets, dtype=np.float64)
    rdm = 1 - np.corrcoef(t)
    np.fill_diagonal(rdm, 0)
    return rdm


@torch.no_grad()
def embeddings(model, loaders, device):
    """[N, n_prompts] fp32 predictions of `model` for every image of `loaders` (ResidentLoaders in a fixed order),
    through the cached, graph-replayed forward where the trunk cache holds the batch."""
    from functions import _pipeline_core as core
    model.eval()
    fwd = core._CachedForwardGraphs.of(model)
    chunks = []
    for loader in loaders:
        for batch in loader:
            images = batch[1].to(device, non_blocking=True)
            if fwd.usable(loader):
                chunks.append(fwd(images, loader.last_ids_dev))
            else:
                core._announce_ids(model, loader)
                chunks.append(model(images))
    return torch.cat(chunks, 0)


def clip_rsa_over_checkpoints(model, loaders, reference_rdm, files, device, rank=0, world_size=1, output_csv=None,
                              log=print, root=None, evaluator=None, embed_fn=None, n_perm=0, n_boot=0, seed=0,
                              kendall=False):
    """-> (rows, per-rank stats) on rank 0 | None.  `model`: CLIPHBA with its adapters applied (weights of the
    checkpoints are loaded with strict=False exactly as NEW:1159 does); `loaders`: ResidentLoaders whose concatenation
    is the image set in the order of `reference_rdm`'s rows.  `evaluator` / `embed_fn` default to the libhba ones
    (hba.rsa.RSAEvaluator, `embeddings`); the world-2 `gloo` test of the sharding passes CPU stand-ins.
    n_perm > 0 adds PERMUTATION_COLUMNS (RSAEvaluator.permutation_test), n_boot > 0 adds BOOTSTRAP_COLUMNS
    (RSAEvaluator.bootstrap, 95 % percentile interval); `seed` seeds both, so every checkpoint sees the same
    permutations and resamples.  kendall=True adds KENDALL_COLUMNS (RSAEvaluator.kendall_tau)."""
    if evaluator is None:
        from .rsa import RSAEvaluator
        evaluator = RSAEvaluator(reference_rdm, device)
    embed_fn = embed_fn or embeddings
    on_cuda = torch.device(device).type == "cuda"
    rows, t_emb, t_rsa = [], 0.0, 0.0
    for path in files[rank::world_size]:
        state = torch.load(path, map_location="cpu")
        missing = model.load_state_dict(state, strict=False)
        if missing.unexpected_keys:
            raise RuntimeError(f"{path}: unexpected keys {missing.unexpected_keys[:3]} (adapter placement differs)")
        t0 = time.perf_counter()
        emb = embed_fn(model, loaders, device)
        if on_cuda:
            torch.cuda.synchronize(device)
        t1 = time.perf_counter()
        rho, p, _ = evaluator(emb, want_rdm=False)
        t2 = time.perf_counter()
        t_emb, t_rsa = t_emb + (t1 - t0), t_rsa + (t2 - t1)
        rel = os.path.relpath(path, root) if root else path
        rows.append({"checkpoint": rel, "run": os.path.basename(os.path.dirname(os.path.dirname(path))) or ".",
                     "epoch": int(_EPOCH.search(path).group(1)), "behavioral_rsa_rho": rho,
                     "behavioral_rsa_p_value": p})
        if n_perm > 0:
            rows[-1]["behavioral_rsa_p_perm"] = evaluator.permutation_test(emb, n_perm=n_perm, seed=seed)[1]
        if n_boot > 0:
            (lo, hi), _, valid = evaluator.bootstrap(emb, n_boot=n_boot, seed=seed)
            rows[-1].update(behavioral_rsa_ci_low=lo, behavioral_rsa_ci_high=hi, behavioral_rsa_boot_valid=valid)
        if kendall:
            tau_a, tau_b = evaluator.kendall_tau(emb)
            rows[-1].update(behavioral_rsa_tau_a=tau_a, behavioral_rsa_tau_b=tau_b)
        if log is not None:
            log(f"[rank {rank}] {rel}: rho {rho:.6f}")
    stats = {"rank": rank, "checkpoints": len(rows), "embed_s": t_emb, "rsa_tail_s": t_rsa}
    if world_size > 1:
        import torch.distributed as dist
        gathered = [None] * world_size
        dist.all_gather_object(gathered, (rows, stats))
        rows = [r for part, _ in gathered for r in part]
        stats = [s for _, s in gathered]
    else:
        stats = [stats]
    if rank != 0:
        return None
    rows.sort(key=lambda r: (r["checkpoint"]))
    if output_csv:
        import pandas as pd
        os.makedirs(os.path.dirname(os.path.abspath(output_csv)), exist_ok=True)
        columns = (list(RESULT_COLUMNS) + (list(PERMUTATION_COLUMNS) if n_perm > 0 else [])
                   + (list(BOOTSTRAP_COLUMNS) if n_boot > 0 else []) + (list(KENDALL_COLUMNS) if kendall else []))
        pd.DataFrame(rows, columns=columns).to_csv(output_csv, index=False)
    return rows, stats
