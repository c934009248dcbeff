"""ORACLE (test infrastructure only; nothing under vit-project_b200/ imports this).

`run_behavioral_training(config)` of BOTH CLIP-HBA pipelines, end to end on the CPU, reference and product side by
side - the unit a sweep shards (SURVEY 8e), from the csv / image files to the result CSV:

  reference arm : the reference's OWN `run_behavioral_training` of BASE (Training/functions/
                  cvpr_train_behavior_things_pipeline_baseline.py:707-823) and of NEW (Training/functions/
                  new_cvpr_train_behavior_things_pipeline.py:1066-1227) with `config['cuda'] = 2` (its CPU branch,
                  NEW:1143-1144), imported unmodified through oracle/ref_loader.py on the restated CLIP towers
                  (oracle/clip_ref.py, "ViT-tiny/14": 3 vision / 2 text blocks).  Replaced, outside the arithmetic:
                  NEW's `save_dora_parameters` (NEW:665-669 hard-codes ViT-L/14's block numbers) by the located-layer
                  writer of the same file format, and `torch.load` defaults to `weights_only=False` (NEW:110 predates
                  torch 2.6).
  product arm   : this repo's `functions.*.run_behavioral_training` as shipped - datasets and the THINGS transform,
                  resident loaders, CLIPHBA on the plug-in `clip`, hba.DoRALayer, the libhba engine (forward, live
                  sub-graph backward, frozen-trunk cache), fused MSE / NaN guard, FusedAdamW, hba.rsa, checkpoints,
                  resume - in the fp32 parity mode, with libhba's entry points served by the CPU restatement of the
                  C-ABI (oracle/libhba_ref.py: `emulated_device()`) and `select_device` answering "cpu".

Both arms read the same files: PNG images, the SPoSE-layout csv (66 target columns), the 8-image inference csv,
RDM48_triplet.mat, and one seeded checkpoint under a private HOME.  Sequence: a 3-epoch baseline run (BASE), then a
perturbation condition (NEW: random targets in epoch 3, resumed from the baseline's epoch-2 checkpoints, run to
epoch 4), a label-shuffle condition from the same checkpoints, and a condition that perturbs epoch 1 (uniform images;
nothing to resume: its DoRA matrices are drawn after the model construction, like the baseline's).  Compared:
every result CSV, the DoRA checkpoint of the last epoch, the optimizer step count and the RNG / generator state of the
last random-state checkpoint.  Two more baseline runs adapt 2 + 2 and 3 + 2 blocks (the general placement path of hba.engine).

    python oracle/clip_pipeline_exec.py --arm reference --out tests/golden/clip_pipeline_exec.json
    python oracle/clip_pipeline_exec.py --arm product --out /tmp/product.json
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import tempfile

# both arms run on the CPU whatever the host has: a visible GPU would add CUDA RNG states to the random-state
# checkpoints, whose keys are compared with tests/golden/clip_pipeline_exec.json
os.environ["CUDA_VISIBLE_DEVICES"] = ""

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "vit-project_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_IMAGES, N_RSA, BATCH = 14, 8, 4


def write_dataset(root):
    import pandas as pd
    import scipy.io
    from PIL import Image
    rng = np.random.default_rng(0)
    img_dir = os.path.join(root, "imgs")
    os.makedirs(img_dir)

    def make(prefix, n):
        names = []
        for i in range(n):
            name = f"{prefix}{i:03d}.png"
            Image.fromarray(rng.integers(0, 255, (24, 24, 3), dtype=np.uint8)).save(os.path.join(img_dir, name))
            names.append(name)
        return names
    tr, rs = make("train", N_IMAGES), make("rsa", N_RSA)
    cols = {"image": tr}
    for k in range(66):
        cols[f"dim{k}"] = rng.standard_normal(N_IMAGES) * 9.5 + 5.75
    pd.DataFrame(cols).to_csv(os.path.join(root, "train.csv"))
    cols = {"image": rs}
    for k in range(66):
        cols[f"dim{k}"] = rng.standard_normal(N_RSA)
    pd.DataFrame(cols).to_csv(os.path.join(root, "rsa.csv"))
    rdm = 1 - np.corrcoef(rng.standard_normal((N_RSA, 66)))
    np.fill_diagonal(rdm, 0)
    scipy.io.savemat(os.path.join(root, "RDM48_triplet.mat"), {"RDM48_triplet": rdm})
    return img_dir


def _sha(t):
    if isinstance(t, torch.Tensor):
        t = t.detach().cpu().contiguous().numpy()
    return hashlib.sha256(np.ascontiguousarray(t).tobytes()).hexdigest()[:16]


def summarise(run_dir, res_csv, dora_dir, rand_dir):
    text = open(res_csv).read()
    rows = [r.split(",") for r in text.replace("\r\n", "\n").strip().split("\n")]
    last = int(rows[-1][0])
    dora = torch.load(os.path.join(dora_dir, f"epoch{last}_dora_params.pth"))
    ck = torch.load(os.path.join(rand_dir, f"epoch{last}_random_states.pth"), weights_only=False)
    return {"csv": text, "last_epoch": last,
            "dora_keys": sorted(dora), "dora": {k: [float(v.double().sum()), float(v.double().abs().max())] for k, v in dora.items()},
            "optimizer_steps": sorted({float(s["step"]) for s in ck["optimizer_state_dict"]["state"].values()}),
            "n_optimizer_tensors": len(ck["optimizer_state_dict"]["state"]),
            "torch_rng_sha": _sha(ck["torch_rng_state"]), "generator_sha": _sha(ck["dataloader_generator_state"]),
            "numpy_rng_sha": _sha(ck["numpy_rng_state"][1]), "random_state_keys": sorted(ck),
            "files": sorted(f for f in os.listdir(run_dir) if not f.startswith("training_log_"))}


def run_arm(arm):
    home = tempfile.mkdtemp(prefix="hba_exec_home_")
    os.environ["HOME"] = home
    os.environ["HBA_SYNTHETIC_OK"] = "1"
    from oracle import clip_ref
    # one checkpoint file for both arms (either `_download` returns a cached file as it is)
    os.makedirs(os.path.join(home, ".cache", "clip"))
    torch.save(clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1), os.path.join(home, ".cache", "clip", "ViT-tiny-14.pt"))
    root = tempfile.mkdtemp(prefix="hba_exec_data_")
    img_dir = write_dataset(root)
    stack = None
    if arm == "reference":
        import functools
        from oracle import ref_loader
        real_load = torch.load
        torch.load = functools.wraps(real_load)(lambda *a, **k: real_load(*a, **{"weights_only": False, **k}))
        NEW, BASE = ref_loader.load_reference()
        NEW.save_dora_parameters = lambda m, path, epoch, logger=None: ref_loader._save_dora_parameters_stub(m, path, epoch, 2, 1)
        cuda_flag = 2          # the reference's CPU branch (NEW:1143-1144)
    else:
        import contextlib
        import hba
        import functions.cvpr_train_behavior_things_pipeline_baseline as BASE
        import functions.new_cvpr_train_behavior_things_pipeline as NEW
        from oracle.libhba_ref import emulated_device
        hba.set_precision("fp32")
        stack = contextlib.ExitStack()
        ref_lib = stack.enter_context(emulated_device())
        BASE.select_device = NEW.select_device = lambda flag: torch.device("cpu")
        cuda_flag = 0
    common = {"csv_file": f"{root}/train.csv", "img_dir": img_dir, "inference_csv_file": f"{root}/rsa.csv",
              "RDM48_triplet_dir": f"{root}/RDM48_triplet.mat", "backbone": "ViT-tiny/14", "batch_size": BATCH,
              "lr": 3e-3, "random_seed": 1, "vision_layers": 2, "transformer_layers": 1, "rank": 8, "cuda": cuda_flag,
              "criterion": torch.nn.MSELoss()}
    out = {"arm": arm, "runs": {}}
    try:
        b = f"{root}/base"
        os.makedirs(b)
        BASE.run_behavioral_training(dict(common, epochs=3, train_portion=0.8, early_stopping_patience=100,
                                          checkpoint_path=f"{b}/model.pth", training_res_path=f"{b}/res.csv",
                                          dora_parameters_path=f"{b}/dora", random_state_path=f"{b}/rand"))
        out["runs"]["baseline"] = summarise(b, f"{b}/res.csv", f"{b}/dora", f"{b}/rand")
        # (the last condition perturbs epoch 1: nothing is resumed, its DoRA matrices are drawn from the seeded RNG
        # after the model construction - NEW:1154-1168 finds no epoch-0 checkpoint - exactly like the baseline's)
        for name, kind, dist, run, epochs in (("random_target", "random_target", "target", 3, 4),
                                              ("label_shuffle", "label_shuffle", "normal", 3, 4),
                                              ("uniform_images_from_scratch", "uniform_images", "target", 1, 2)):
            d = f"{root}/{name}"
            os.makedirs(d)
            NEW.run_behavioral_training(dict(
                common, epochs=epochs, early_stopping_patience=100, checkpoint_path=f"{d}/model.pth",
                training_res_path=f"{d}/res.csv", dora_parameters_path=f"{d}/dora", random_state_path=f"{d}/rand",
                baseline_dora_directory=f"{b}/dora", baseline_random_state_path=f"{b}/rand",
                baseline_split_indices_path=f"{b}/rand/dataset_split_indices.pth", training_run=run,
                resume_from_epoch=run - 1, perturb_type=kind, perturb_length=1, perturb_distribution=dist,
                perturb_seed=42, previous_training_res_path=f"{b}/res.csv"))
            out["runs"][name] = summarise(d, f"{d}/res.csv", f"{d}/dora", f"{d}/rand")
        # another adapter placement than the drivers' 2 + 1: every block of the miniature adapted (NEW:484-513 is general)
        # (2 + 2 in the fp32 parity mode: the text tower's general path; 3 + 2 in the bf16 mode: at the pipeline's
        # 224-pixel images the vision tower has T = 257 tokens, beyond the fp32 form of the full attention backward)
        for name, nv, nt, mode in (("baseline_2p2", 2, 2, "fp32"), ("baseline_3p2", 3, 2, "bf16")):
            if stack is not None:
                hba.set_precision(mode)
            g3 = f"{root}/{name}"
            os.makedirs(g3)
            BASE.run_behavioral_training(dict(common, vision_layers=nv, transformer_layers=nt, epochs=2, train_portion=0.8,
                                              early_stopping_patience=100, checkpoint_path=f"{g3}/model.pth",
                                              training_res_path=f"{g3}/res.csv", dora_parameters_path=f"{g3}/dora",
                                              random_state_path=f"{g3}/rand"))
            out["runs"][name] = summarise(g3, f"{g3}/res.csv", f"{g3}/dora", f"{g3}/rand")
        if stack is not None:
            hba.set_precision("fp32")
        if stack is not None:
            calls = ref_lib.calls
            out["c_abi_calls"] = {n: calls.count(n) for n in sorted(set(calls))}
            # RSA at scale over the checkpoints the baseline left behind (hba.rsa_scale, BASELINE config 5), restricted
            # to the inference set and its own reference RDM: must give back the rho train_model logged per epoch
            import logging
            import scipy.io
            import functions._pipeline_core as core
            from hba import rsa_scale
            from hba.data import ResidentLoader, ResidentStore
            os.environ["HBA_CONSTRUCTOR_RNG"] = "0"
            model = core.build_model(dict(common), torch.device("cpu"), logging.getLogger("exec_rsa_scale"))
            inf = core.ThingsInferenceDataset(common["inference_csv_file"], img_dir, common["RDM48_triplet_dir"])
            loader = ResidentLoader(ResidentStore(inf, "cpu"), BATCH, shuffle=False, dataset=inf)
            core.enable_trunk_cache(model, len(inf))
            rows, stats = rsa_scale.clip_rsa_over_checkpoints(
                model, [loader], scipy.io.loadmat(common["RDM48_triplet_dir"])["RDM48_triplet"],
                rsa_scale.find_dora_checkpoints(f"{b}/dora"), "cpu", log=None, root=b)
            out["rsa_over_checkpoints"] = rows
    finally:
        if stack is not None:
            stack.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", choices=["reference", "product"], required=True)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    torch.set_num_threads(max(1, min(4, os.cpu_count() or 1)))
    import contextlib
    import io
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):          # (the pipelines log every line to stdout as well as to their file)
        res = run_arm(a.arm)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"{a.arm}: " + ", ".join(f"{k}: epochs up to {v['last_epoch']}" for k, v in res["runs"].items()))


if __name__ == "__main__":
    main()
