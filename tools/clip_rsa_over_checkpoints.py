#!/usr/bin/env python
"""RSA at scale for CLIP-HBA (BASELINE.json configs[4]; hba.rsa_scale.clip_rsa_over_checkpoints): RDM + Spearman rho
of the 66-D embeddings of ALL images (1,854 in the reference's files) for every `epoch{N}_dora_params.pth` under a
checkpoint tree (a baseline run and / or the output tree of a sweep), checkpoints sharded across ranks.

  torchrun --nproc_per_node=8 tools/clip_rsa_over_checkpoints.py --checkpoints /runs/sweep_out \
      --csv-file train.csv --inference-csv-file rsa.csv --img-dir imgs [--rdm ref_rdm.npy] --output-csv rsa_scale.csv

Reference RDM: `--rdm` (.npy or .mat with one square matrix), else 1 - corrcoef of the 66-D behavioural embedding in
the two CSV files (rows in the order train csv, then inference csv) - what RDM48_triplet is for the 48-image subset.
The last stdout line is a JSON record with checkpoints/s (wall clock, max over ranks, cache fill included).
--permutations N adds the Mantel p-value column behavioral_rsa_p_perm, --bootstrap N the stimulus-bootstrap 95 %
interval (behavioral_rsa_ci_low / _ci_high) and the number of valid replicates (behavioral_rsa_boot_valid); --seed
seeds both, identically for every checkpoint.  --kendall adds Kendall's tau-a and tau-b of each model RDM against the
reference (behavioral_rsa_tau_a / _tau_b).  Without these flags the CSV has the columns of
hba.rsa_scale.RESULT_COLUMNS.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "vit-project_b200")]


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--checkpoints", required=True, help="directory tree holding epoch*_dora_params.pth files")
    ap.add_argument("--csv-file", required=True)
    ap.add_argument("--inference-csv-file", required=True)
    ap.add_argument("--img-dir", required=True)
    ap.add_argument("--rdm", default="")
    ap.add_argument("--output-csv", default="")
    ap.add_argument("--backbone", default="ViT-L/14")
    ap.add_argument("--vision-layers", type=int, default=2)
    ap.add_argument("--transformer-layers", type=int, default=1)
    ap.add_argument("--rank", type=int, default=32, dest="dora_rank")
    ap.add_argument("--batch-size", type=int, default=32)
    ap.add_argument("--limit", type=int, default=0)
    ap.add_argument("--permutations", type=int, default=0, help="Mantel permutations per checkpoint (0: none)")
    ap.add_argument("--bootstrap", type=int, default=0, help="stimulus-bootstrap replicates per checkpoint (0: none)")
    ap.add_argument("--seed", type=int, default=0, help="seed of the permutations and resamples")
    ap.add_argument("--kendall", action="store_true",
                    help="add Kendall's tau-a and tau-b columns (tau-a: preferred when either RDM has ties)")
    a = ap.parse_args(argv)
    import numpy as np
    import pandas as pd
    import torch
    import torch.distributed as dist
    from functions import _pipeline_core as core
    from hba import rsa_scale
    from hba.data import ResidentLoader, ResidentStore
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    t_start = time.perf_counter()
    import logging
    logger = logging.getLogger("clip_rsa_scale")
    logger.addHandler(logging.NullHandler())
    config = {"backbone": a.backbone, "vision_layers": a.vision_layers, "transformer_layers": a.transformer_layers,
              "rank": a.dora_rank}
    # (every DoRA tensor comes from a checkpoint here: the random draws of the model construction decide nothing)
    os.environ.setdefault("HBA_CONSTRUCTOR_RNG", "0")
    model = core.build_model(config, device, logger).to(device)
    train_set = core.ThingsDataset(csv_file=a.csv_file, img_dir=a.img_dir)
    rsa_set = core.ThingsInferenceDataset(inference_csv_file=a.inference_csv_file, img_dir=a.img_dir,
                                          RDM48_triplet_dir=None)
    stores = [ResidentStore(train_set, device), ResidentStore(rsa_set, device)]
    loaders = [ResidentLoader(s, a.batch_size, shuffle=False) for s in stores]
    n_images = sum(len(s) for s in stores)
    core.enable_trunk_cache(model, n_images)
    if a.rdm:
        if a.rdm.endswith(".npy"):
            ref = np.load(a.rdm)
        else:
            import scipy.io
            mats = [v for k, v in scipy.io.loadmat(a.rdm).items() if not k.startswith("__")]
            ref = next(m for m in mats if getattr(m, "ndim", 0) == 2 and m.shape[0] == m.shape[1])
    else:
        cols = [pd.read_csv(f, index_col=0).iloc[:, 1:67].to_numpy(dtype=np.float64)
                for f in (a.csv_file, a.inference_csv_file)]
        ref = rsa_scale.reference_rdm_from_targets(np.concatenate(cols, 0))
    if ref.shape[0] != n_images:
        raise SystemExit(f"reference RDM is {ref.shape[0]} x {ref.shape[0]} but the image set has {n_images} images")
    files = rsa_scale.find_dora_checkpoints(a.checkpoints)
    if a.limit:
        files = files[:a.limit]
    if not files:
        raise SystemExit(f"no epoch*_dora_params.pth under {a.checkpoints}")
    t_setup = time.perf_counter() - t_start
    res = rsa_scale.clip_rsa_over_checkpoints(model, loaders, ref, files, device, rank=rank, world_size=world,
                                              output_csv=a.output_csv or None, log=None, root=a.checkpoints,
                                              n_perm=a.permutations, n_boot=a.bootstrap, seed=a.seed,
                                              kendall=a.kendall)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t_start
    if world > 1:
        t = torch.tensor([wall], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall = float(t)
    if rank == 0:
        rows, stats = res
        work = wall - t_setup
        print(json.dumps({"metric": "CLIP-HBA RSA at scale: checkpoints/s", "n_gpus": world, "checkpoints": len(rows),
                          "images_per_checkpoint": n_images, "pairs_per_checkpoint": n_images * (n_images - 1) // 2,
                          "wall_s": wall, "setup_s": t_setup, "checkpoints_per_s": len(rows) / max(work, 1e-9),
                          "checkpoints_per_s_incl_setup": len(rows) / wall,
                          "per_rank": stats,
                          "rho_first_last": [rows[0]["behavioral_rsa_rho"], rows[-1]["behavioral_rsa_rho"]],
                          "what": "per checkpoint: load DoRA tensors, cached + graph-replayed forward of every image "
                                  "(frozen trunk from the HBM cache; the first checkpoint of a rank fills it), "
                                  "hba_rdm_spearman (RDM f64 -> keys -> radix sort -> tie-averaged ranks -> rho)"}))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
