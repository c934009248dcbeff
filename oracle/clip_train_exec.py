"""ORACLE (test infrastructure only; nothing under vit-project_b200/ imports this).

The epoch loops of the two CLIP-HBA pipelines EXECUTED on the CPU, reference and product side by side:

  reference arm : the reference's OWN `train_model`, `evaluate_model`, `behavioral_RSA`, `shuffle_targets`,
                  `save_random_states`, `load_random_states` of NEW (Training/functions/
                  new_cvpr_train_behavior_things_pipeline.py:88-134, 584-654, 696-1063) and `train_model` of BASE
                  (Training/functions/cvpr_train_behavior_things_pipeline_baseline.py:612-704), imported unmodified
                  through oracle/ref_loader.py.  Two things are replaced, both outside the arithmetic:
                  `save_dora_parameters` (NEW:665-669 hard-codes ViT-L/14's block numbers 22 / 23 / 11; BASE imports
                  it from the un-vendored `src.models.clip_hba_utils`) writes the stand-in model's state dict to the
                  same file name, and `torch.load` defaults to `weights_only=False` (the reference's
                  `load_random_states`, NEW:110, was written for torch < 2.6 and unpickles NumPy RNG states).
  product arm   : `functions.new_cvpr_train_behavior_things_pipeline.train_model` /
                  `functions.cvpr_train_behavior_things_pipeline_baseline.train_model` of this repo - the host
                  orchestration as shipped (TrainStep, device-side NaN guard and loss accumulation, Perturbation,
                  ResidentStore / ResidentLoader on the "cpu" device, CheckpointWriter, CSV bootstrap, early stopping)
                  - with the two libhba entry points the generic (non-fused) path touches replaced by torch / NumPy /
                  SciPy stand-ins: `hba.ops.nonfinite_flag` and `hba.rsa.RSAEvaluator`.

Both arms train the same tiny stand-in network (Linear 108 -> 66 on 3 x 6 x 6 "images"; one training image is NaN,
so the NaN guard of NEW:989-998 fires in every un-perturbed epoch) on the same files and RNG streams.  What is
compared: the result CSV text, the number of epochs run (early stopping, counter frozen inside the perturbation
window, NEW:1042-1063), the final parameters, the optimizer / RNG / DataLoader-generator state of the last random-state
checkpoint, and the files written.  The device arithmetic (CLIP towers, DoRA, fused AdamW, the RSA kernels) is NOT
exercised here - that is the GPU tests' job.

    python oracle/clip_train_exec.py --arm reference --out tests/golden/clip_train_exec.json   # regenerate the golden
    python oracle/clip_train_exec.py --arm product --out /tmp/product.json
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import random
import sys
import tempfile

# both arms run on the CPU whatever the host has: a visible GPU would add CUDA RNG states to the random-state
# checkpoints, whose keys are compared with tests/golden/clip_train_exec.json
os.environ["CUDA_VISIBLE_DEVICES"] = ""

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "vit-project_b200")
for _p in (PKG, ROOT):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_TRAIN, N_TEST, N_RSA, BATCH = 22, 9, 10, 8

# (name, pipeline, keyword arguments of train_model, learning rate, resume spec)
CASES = [
    ("random_target_window2", "NEW", dict(epochs=7, training_run=2, perturb_length=2, perturb_seed=42,
                                          perturb_distribution="target", perturb_type="random_target",
                                          early_stopping_patience=2), 3e-2, None),
    ("label_shuffle_normal", "NEW", dict(epochs=4, training_run=1, perturb_length=1, perturb_seed=7,
                                         perturb_distribution="normal", perturb_type="label_shuffle",
                                         early_stopping_patience=10), 1e-2, None),
    ("image_noise", "NEW", dict(epochs=4, training_run=3, perturb_length=1, perturb_seed=0,
                                perturb_distribution="target", perturb_type="image_noise",
                                early_stopping_patience=10), 1e-2, None),
    ("uniform_images_frozen_patience", "NEW", dict(epochs=12, training_run=2, perturb_length=3, perturb_seed=1,
                                                   perturb_distribution="target", perturb_type="uniform_images",
                                                   early_stopping_patience=1), 2e-1, None),
    # resumes: from another run's checkpoints into a new CSV (pre-populated rows, NEW:816-834), then in place
    ("resume_other_file", "NEW", dict(epochs=6, training_run=4, perturb_length=1, perturb_seed=42,
                                      perturb_distribution="normal", perturb_type="random_target",
                                      early_stopping_patience=10), 3e-2, ("random_target_window2", 3, False)),
    ("resume_same_file", "NEW", dict(epochs=8, training_run=4, perturb_length=1, perturb_seed=42,
                                     perturb_distribution="normal", perturb_type="random_target",
                                     early_stopping_patience=10), 3e-2, ("resume_other_file", 5, True)),
    ("baseline_early_stop", "BASE", dict(epochs=30, early_stopping_patience=2, vision_layers=2,
                                         transformer_layers=1), 2e-1, None),
]


# ------------------------------------------------------------------------------- the shared problem
class ListDataset(torch.utils.data.Dataset):
    def __init__(self, items, **attrs):
        self.items = items
        self.__dict__.update(attrs)

    def __len__(self):
        return len(self.items)

    def __getitem__(self, i):
        return self.items[i]


class StandIn(torch.nn.Module):
    """images [B, 3, 6, 6] -> 66 'SPoSE' predictions."""

    def __init__(self):
        super().__init__()
        g = torch.Generator().manual_seed(7)
        self.fc = torch.nn.Linear(108, 66)
        with torch.no_grad():
            self.fc.weight.copy_(torch.randn(66, 108, generator=g) * 0.05)
            self.fc.bias.zero_()

    def forward(self, x):
        return self.fc(x.flatten(1))


def make_problem(tmp):
    import scipy.io
    g = torch.Generator().manual_seed(0)
    n = N_TRAIN + N_TEST
    images = torch.randn(n, 3, 6, 6, generator=g)
    truth = torch.randn(108, 66, generator=g) * 0.6
    targets = images.flatten(1) @ truth + torch.randn(n, 66, generator=g) * 4.0 + 5.75
    clean5 = images[5].clone()
    images[5] = float("nan")          # a training image: NEW:989-998 skips its batch in un-perturbed epochs
    rsa_images = torch.randn(N_RSA, 3, 6, 6, generator=g)
    human = 1 - np.corrcoef(torch.randn(N_RSA, 66, generator=g).numpy().astype(np.float64))
    np.fill_diagonal(human, 0)
    mat = os.path.join(tmp, "RDM48_triplet.mat")
    scipy.io.savemat(mat, {"RDM48_triplet": human})
    train = ListDataset([(f"tr{i}", images[i], targets[i]) for i in range(N_TRAIN)])
    # (BASE:644-659 has no NaN guard: its case trains on the same set with the NaN image restored)
    train_clean = ListDataset([(f"tr{i}", clean5 if i == 5 else images[i], targets[i]) for i in range(N_TRAIN)])
    test = ListDataset([(f"te{i}", images[N_TRAIN + i], targets[N_TRAIN + i]) for i in range(N_TEST)])
    rsa = ListDataset([(f"rs{i}", rsa_images[i]) for i in range(N_RSA)], RDM48_triplet_dir=mat)
    tvals = targets.numpy().astype("float32")
    return train, train_clean, test, rsa, np.mean(tvals), np.std(tvals)      # mean / std as NEW:1098-1099 computes them


def seed_all(seed):
    torch.manual_seed(seed)
    random.seed(seed)
    np.random.seed(seed)


def _digest(t):
    if isinstance(t, torch.Tensor):
        t = t.detach().cpu().contiguous().numpy()
    return hashlib.sha256(np.ascontiguousarray(t).tobytes()).hexdigest()[:16]


def _save_state_stub(model, path, epoch, *_, **__):
    os.makedirs(path, exist_ok=True)
    torch.save({k: v.detach().cpu().clone() for k, v in model.state_dict().items()},
               os.path.join(path, f"epoch{epoch + 1}_dora_params.pth"))


# ------------------------------------------------------------------------------- stand-ins of the product arm
class _NumpyRSA:
    """hba.rsa.RSAEvaluator's contract (-> rho, p, rdm) on NumPy / SciPy: the device tail is not under test here."""

    def __init__(self, reference_rdm, device="cpu"):
        self.ref = np.asarray(reference_rdm, dtype=np.float64)

    def __call__(self, emb, want_rdm=True):
        from scipy.stats import spearmanr
        rdm = 1 - np.corrcoef(emb.detach().cpu().numpy())
        np.fill_diagonal(rdm, 0)
        iu = np.triu_indices_from(self.ref, k=1)
        rho, p = spearmanr(self.ref[iu], rdm[iu])
        return rho, p, rdm


def _nonfinite_flag_cpu(x, flag):
    flag += int(not bool(torch.isfinite(x).all()))


# ------------------------------------------------------------------------------- arms
def _modules(arm):
    if arm == "reference":
        from oracle import ref_loader
        import functools
        real_load = torch.load
        torch.load = functools.wraps(real_load)(lambda *a, **k: real_load(*a, **{"weights_only": False, **k}))
        NEW, BASE = ref_loader.load_reference()
        NEW.save_dora_parameters = lambda m, path, epoch, logger=None: _save_state_stub(m, path, epoch)
        BASE.save_dora_parameters = _save_state_stub
        return NEW, BASE
    import hba.ops
    import hba.rsa
    import functions._pipeline_core as core
    import functions.cvpr_train_behavior_things_pipeline_baseline as BASE
    import functions.new_cvpr_train_behavior_things_pipeline as NEW
    hba.ops.nonfinite_flag = _nonfinite_flag_cpu
    hba.rsa.RSAEvaluator = _NumpyRSA
    core._RSA_CACHE.clear()
    NEW.save_dora_parameters = lambda m, path, epoch, logger=None: _save_state_stub(m, path, epoch)
    BASE.save_dora_parameters = _save_state_stub
    return NEW, BASE


def _loaders(arm, train, test, rsa, gen):
    if arm == "reference":
        DL = torch.utils.data.DataLoader
        return (DL(train, batch_size=BATCH, shuffle=True, generator=gen), DL(test, batch_size=BATCH, shuffle=False),
                DL(rsa, batch_size=BATCH, shuffle=False))
    from hba.data import ResidentLoader, ResidentStore
    st_tr, st_te, st_rs = (ResidentStore(d, "cpu") for d in (train, test, rsa))
    return (ResidentLoader(st_tr, BATCH, shuffle=True, generator=gen, dataset=train),
            ResidentLoader(st_te, BATCH, shuffle=False, dataset=test),
            ResidentLoader(st_rs, BATCH, shuffle=False, dataset=rsa))


def run_arm(arm):
    NEW, BASE = _modules(arm)
    out = {"arm": arm, "cases": {}}
    with tempfile.TemporaryDirectory() as tmp:
        train, train_clean, test, rsa, mean, std = make_problem(tmp)
        out["mean_std"] = [float(mean), float(std)]
        logger = NEW.setup_logger(os.path.join(tmp, "log.txt"))
        for h in [h for h in logger.handlers if not hasattr(h, "baseFilename")]:
            logger.removeHandler(h)        # (keep the file handler only: the harness prints one summary line)
        for name, pipe, kw, lr, resume in CASES:
            d = os.path.join(tmp, name)
            seed_all(1)
            model = StandIn()
            opt = torch.optim.AdamW(model.parameters(), lr=lr)
            gen = torch.Generator()
            gen.manual_seed(1)
            tl, el, rl = _loaders(arm, train_clean if pipe == "BASE" else train, test, rsa, gen)
            crit = torch.nn.MSELoss()
            common = dict(logger=logger, dora_parameters_path=os.path.join(d, "dora"),
                          random_state_path=os.path.join(d, "rand"), dataloader_generator=gen)
            res = os.path.join(d, "res.csv")
            os.makedirs(d, exist_ok=True)
            if pipe == "BASE":
                BASE.train_model(model, tl, el, rl, torch.device("cpu"), opt, crit, training_res_path=res, **kw, **common)
            else:
                extra = {}
                if resume is not None:
                    src, epoch, same_file = resume
                    sd = os.path.join(tmp, src)
                    if same_file:      # continue the earlier case's own files (NEW:801-814)
                        d, res = sd, os.path.join(sd, "res.csv")
                        common.update(dora_parameters_path=os.path.join(d, "dora"), random_state_path=os.path.join(d, "rand"))
                    model.load_state_dict(torch.load(os.path.join(sd, "dora", f"epoch{epoch}_dora_params.pth")))
                    ok = NEW.load_random_states(os.path.join(sd, "rand"), epoch, optimizer=opt, dataloader_generator=gen,
                                                logger=logger)
                    assert ok
                    extra = dict(resume_from_epoch=epoch, previous_training_res_path=os.path.join(sd, "res.csv"))
                NEW.train_model(model, tl, el, rl, torch.device("cpu"), opt, crit, training_res_path=res, mean=mean,
                                std=std, **kw, **extra, **common)
            text = open(res).read()
            rows = [r.split(",") for r in text.replace("\r\n", "\n").strip().split("\n")]
            last = int(rows[-1][0])
            ck = torch.load(os.path.join(d, "rand", f"epoch{last}_random_states.pth"), weights_only=False)
            steps = sorted({float(s["step"]) for s in ck["optimizer_state_dict"]["state"].values()})
            out["cases"][name] = {
                "csv": text, "last_epoch": last, "n_rows": len(rows) - 1,
                "params": {k: [float(v.double().sum()), float(v.double().abs().max())] for k, v in model.state_dict().items()},
                "params_sha": {k: _digest(v) for k, v in model.state_dict().items()},
                "optimizer_steps": steps, "checkpoint_epoch": int(ck["epoch"]),
                "exp_avg_sha": [_digest(s["exp_avg"]) for s in ck["optimizer_state_dict"]["state"].values()],
                "torch_rng_sha": _digest(ck["torch_rng_state"]), "numpy_rng_sha": _digest(ck["numpy_rng_state"][1]),
                "python_rng_sha": hashlib.sha256(repr(ck["python_rng_state"]).encode()).hexdigest()[:16],
                "generator_sha": _digest(ck["dataloader_generator_state"]),
                "random_state_keys": sorted(ck), "files": sorted(os.listdir(os.path.join(d, "dora"))
                                                                + os.listdir(os.path.join(d, "rand"))),
            }
        for h in list(logger.handlers):
            h.close()
            logger.removeHandler(h)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", choices=["reference", "product"], required=True)
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    torch.set_num_threads(1)      # same summation order in both arms whatever the host
    res = run_arm(a.arm)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"{a.arm}: " + ", ".join(f"{k}: {v['n_rows']} rows" for k, v in res["cases"].items()))


if __name__ == "__main__":
    main()
