"""CPU tests of the ViT epoch loop / single-epoch perturbation measurement host logic (hba.vit_train;
reference VIT = Training/vit_training/baseline/train_vit_sgd.py, MEAS = Training/vit_training/single_epoch/
measure_single_epoch_perturbation_effect.py):

  * golden vectors written by the reference's own classes / functions / shipped CSVs
    (tests/golden/vit_measure.json, oracle/make_vit_measure_golden.py), and the reference classes directly
    where /root/reference is mounted;
  * the loader order against torch's DataLoader + DistributedSampler;
  * the whole orchestration (checkpoint N-1 reload, perturbed epoch, schedule step, validation, RSA, result
    row, CSV) with the device trainer replaced by a CPU stand-in of the same interface - it must then equal
    the oracle restatement `oracle.vit_measure_ref.measure_ref` exactly;
  * the collective tails on a world-size-2 `gloo` group.
No libhba compute call is made here; the GPU parity of the same functions is tests/test_gpu_vit_measure.py."""
import json
import os
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "vit_measure.json")))
pytestmark = pytest.mark.timeout(900)      # DataLoader workers / spawned ranks: a hang must fail, not stall the suite


def _vt():
    from hba import vit_train
    return vit_train


# ------------------------------------------------------------------------------- goldens of the reference
@pytest.mark.parametrize("seed", [42, 7])
def test_label_perturbations_match_reference_goldens(seed):
    vt = _vt()
    labels = torch.tensor(GOLD["labels"])
    assert vt.perturbed_labels(labels, "label_shuffle", 10, seed).tolist() == GOLD[f"label_shuffle_seed{seed}"]
    assert vt.perturbed_labels(labels, "target_noise", 10, seed).tolist() == GOLD[f"target_noise_seed{seed}"]
    assert vt.perturbed_labels(labels, None, 10, seed) is labels
    base = [(i, l) for i, l in enumerate(GOLD["labels"])]
    sh, tn = vt.ShuffledLabelsDataset(base, shuffle_seed=seed), vt.TargetNoiseDataset(base, 10, noise_seed=seed)
    assert [int(sh[i][1]) for i in range(len(sh))] == GOLD[f"label_shuffle_seed{seed}"]
    assert [int(tn[i][1]) for i in range(len(tn))] == GOLD[f"target_noise_seed{seed}"]
    assert all(sh[i][0] == i and tn[i][0] == i for i in range(len(base)))


def test_target_noise_default_class_count_and_image_transforms():
    vt = _vt()
    labels = torch.tensor(GOLD["labels"])
    assert vt.perturbed_labels(labels, "target_noise").tolist() == GOLD["target_noise_1000_seed42"]
    t = torch.arange(12.0).reshape(3, 2, 2)
    torch.manual_seed(5)
    got = vt.GaussianNoiseTransform(lambda im: im, epsilon=0.25)(t)
    assert got.flatten().tolist() == GOLD["gaussian_eps0.25_seed5"]
    assert float(vt.UniformGrayTransform(lambda im: im)(t).abs().sum()) == GOLD["uniform_gray_sum"] == 0.0


def test_schedule_matches_reference_goldens():
    from hba import vit
    opt = types.SimpleNamespace(param_groups=[{"lr": 0.1}])
    s = vit.CosineAnnealingLRWithWarmup(opt, warmup_epochs=5, max_epochs=100, eta_min=0)
    lrs = []
    for e in range(100):
        if e == 40:   # state round trip in the middle (resume, VIT:322)
            s2 = vit.CosineAnnealingLRWithWarmup(opt, warmup_epochs=1, max_epochs=2)
            s2.load_state_dict(s.state_dict())
            s = s2
        s.step()
        lrs.append(opt.param_groups[0]["lr"])
    assert lrs == pytest.approx(GOLD["schedule_vit"], rel=1e-15, abs=1e-18)
    assert GOLD["schedule_vit"] == GOLD["schedule_meas"]
    assert s.state_dict() == GOLD["schedule_vit_state"]


class _TorchTrainer:
    """CPU stand-in with hba.vit.DataParallelTrainer's interface: torch autograd + torch.optim.SGD."""

    def __init__(self, model, lr=0.1, momentum=0.9, weight_decay=1e-4, process_group=None, use_graph=False):
        self.model = model
        self.opt = torch.optim.SGD(model.parameters(), lr=lr, momentum=momentum, weight_decay=weight_decay)
        self.param_groups = self.opt.param_groups

    def step(self, images, labels):
        self.model.train()
        self.opt.zero_grad()
        out = self.model(images)
        loss = F.cross_entropy(out, labels)
        loss.backward()
        self.opt.step()
        return loss.detach().reshape(1), out.max(1)[1].eq(labels).sum().to(torch.int32).reshape(1)

    def evaluate(self, images, labels):
        self.model.eval()
        with torch.no_grad():
            out = self.model(images)
            return F.cross_entropy(out, labels).reshape(1), out.max(1)[1].eq(labels).sum().to(torch.int32).reshape(1)

    def state_dict(self):
        return self.opt.state_dict()

    def load_state_dict(self, sd):
        self.opt.load_state_dict(sd)


def test_save_checkpoint_format_matches_reference(tmp_path):
    vt = _vt()
    from hba import vit
    lin = torch.nn.Linear(3, 2)
    tr = _TorchTrainer(lin)
    tr.step(torch.ones(4, 3), torch.tensor([0, 1, 0, 1]))
    sched = vit.CosineAnnealingLRWithWarmup(tr, 5, 100)
    d = str(tmp_path)
    vt.save_checkpoint(3, lin, tr, sched, 1.23456789, 2.5, 12.3456789, d, 0)
    vt.save_checkpoint(4, lin, tr, sched, 1.0, 2.0, 50.0, d, 0)
    assert vt.save_checkpoint(5, lin, tr, sched, 1.0, 2.0, 50.0, d, local_rank=1) is None     # VIT:91-92
    assert sorted(os.listdir(d)) == GOLD["checkpoint_files"]
    assert open(os.path.join(d, "training_metrics.csv")).read() == GOLD["metrics_csv"]
    ck = torch.load(os.path.join(d, "checkpoint_epoch_003.pth"), weights_only=False)
    assert sorted(ck.keys()) == GOLD["checkpoint_keys"] and ck["epoch"] == 3
    assert ck["scaler_state_dict"] == GOLD["fresh_grad_scaler_state"]
    latest = torch.load(os.path.join(d, "checkpoint_latest.pth"), weights_only=False)
    assert latest["epoch"] == 4 and torch.equal(latest["model_state_dict"]["weight"], lin.weight.detach())
    # a reference-side torch.optim.SGD loads the optimizer state unchanged
    opt = torch.optim.SGD(torch.nn.Linear(3, 2).parameters(), lr=1.0)
    opt.load_state_dict(ck["optimizer_state_dict"])
    assert opt.param_groups[0]["momentum"] == 0.9 and len(opt.state_dict()["state"]) == 2


def test_result_rows_reproduce_the_shipped_measurements():
    """Data/vit_results/perturbation_effects.csv: columns, condition order and - from the perturbed values and
    the baseline values - the very deltas the reference wrote."""
    vt = _vt()
    assert list(vt.RESULT_COLUMNS) == GOLD["effects_columns"]
    assert list(vt.DEFAULT_PERTURB_EPOCHS) == GOLD["default_perturb_epochs"]
    assert list(vt.PERTURBATION_TYPES) == GOLD["default_perturbation_types"]
    assert [[e, t] for e, t in vt.measurement_conditions()] == GOLD["effects_order"]
    assert (0, "gaussian") not in vt.measurement_conditions([0, 5])                            # MEAS:631-632
    for row in GOLD["effects_rows"]:
        got = vt.assemble_result(row["perturb_epoch"], row["perturbation_type"], row["baseline_loss"],
                                 row["baseline_rsa"], row["perturbed_loss"], row["perturbed_rsa"])
        assert list(got) == GOLD["effects_columns"]
        assert got["delta_loss"] == pytest.approx(row["delta_loss"], rel=1e-12, abs=1e-15)
        assert got["delta_rsa"] == pytest.approx(row["delta_rsa"], rel=1e-12, abs=1e-15)
    none = vt.assemble_result(5, "gaussian", 1.0, 0.25, 2.0, None)                             # MEAS:533-534
    assert none["perturbed_rsa"] == 0.0 and none["delta_rsa"] == -0.25


def test_baseline_row_lookup(tmp_path):
    import pandas as pd
    vt = _vt()
    p = os.path.join(str(tmp_path), "m.csv")
    pd.DataFrame({"epoch": [4, 5], "val_loss": [7.5, 7.129578], "rsa_score": [0.4, 0.4116646782437932]}).to_csv(p, index=False)
    assert vt.baseline_row(p, 5) == (7.129578, 0.4116646782437932)
    assert vt.baseline_row(p, 6) is None


def test_restatement_equals_reference_classes():
    """The product's and the oracle's wrapper classes against the outputs of the reference's own classes stored in
    tests/golden/vit_measure.json, and against those classes themselves (imported with timm stubbed) where the
    reference tree is present."""
    from oracle import make_vit_measure_golden as mk
    from oracle import vit_measure_ref as ref
    vt = _vt()
    gold_base = [(i, l) for i, l in enumerate(GOLD["labels"])]
    for seed in (42, 7):
        for cls in (vt.ShuffledLabelsDataset, ref.ShuffledLabelsRef):
            ds = cls(gold_base, seed)
            assert [int(ds[i][1]) for i in range(len(ds))] == GOLD[f"label_shuffle_seed{seed}"], (cls, seed)
        for cls in (vt.TargetNoiseDataset, ref.TargetNoiseRef):
            ds = cls(gold_base, 10, seed)
            assert [int(ds[i][1]) for i in range(len(ds))] == GOLD[f"target_noise_seed{seed}"], (cls, seed)
    from hba import vit
    for cls in (vit.CosineAnnealingLRWithWarmup, ref.CosineWarmupRef):
        opt = types.SimpleNamespace(param_groups=[{"lr": 0.1}])
        s = cls(opt, 5, 100, eta_min=0)
        lrs = []
        for _ in range(100):
            s.step()
            lrs.append(opt.param_groups[0]["lr"])
        assert lrs == pytest.approx(GOLD["schedule_meas"], rel=1e-15, abs=1e-18), cls
        assert s.state_dict() == GOLD["schedule_meas_state"], cls
    if not os.path.isdir(os.path.join(mk.REF, "Training", "vit_training")):
        return
    MEAS, VIT = mk.load_reference_scripts()
    base = [(torch.full((2,), float(i)), (3 * i + 1) % 13) for i in range(41)]
    for seed in (0, 42):
        a, b, c = MEAS.ShuffledLabelsDataset(base, seed), vt.ShuffledLabelsDataset(base, seed), ref.ShuffledLabelsRef(base, seed)
        assert [a[i][1] for i in range(41)] == [b[i][1] for i in range(41)] == [c[i][1] for i in range(41)]
        a, b, c = MEAS.TargetNoiseDataset(base, 13, seed), vt.TargetNoiseDataset(base, 13, seed), ref.TargetNoiseRef(base, 13, seed)
        assert [int(a[i][1]) for i in range(41)] == [int(b[i][1]) for i in range(41)] == [c[i][1] for i in range(41)]
    for cls in (MEAS.CosineAnnealingLRWithWarmup, VIT.CosineAnnealingLRWithWarmup):
        o1, o2 = types.SimpleNamespace(param_groups=[{"lr": 0.3}]), types.SimpleNamespace(param_groups=[{"lr": 0.3}])
        s1, s2 = cls(o1, 3, 20, eta_min=0.01), ref.CosineWarmupRef(o2, 3, 20, eta_min=0.01)
        for _ in range(20):
            s1.step(), s2.step()
            assert o1.param_groups[0]["lr"] == o2.param_groups[0]["lr"]
        assert s1.state_dict() == s2.state_dict()


# ------------------------------------------------------------------------------- loader order
@pytest.mark.parametrize("world,shuffle", [(1, True), (2, True), (3, False), (2, False)])
def test_sharded_loader_visits_the_distributed_sampler_order(world, shuffle):
    from torch.utils.data import DataLoader, DistributedSampler, TensorDataset
    vt = _vt()
    n = 23
    images = torch.arange(n, dtype=torch.float32).reshape(n, 1, 1, 1).expand(n, 3, 2, 2).contiguous()
    labels = torch.arange(n) % 7
    data = vt.ResidentImageSet(images, labels)
    ds = TensorDataset(images, labels)
    for rank in range(world):
        mine = vt.ShardedLoader(data, 4, world, rank, shuffle=shuffle)
        sampler = DistributedSampler(ds, num_replicas=world, rank=rank, shuffle=shuffle)
        for epoch in (0, 5):
            mine.sampler.set_epoch(epoch)
            sampler.set_epoch(epoch)
            want = list(DataLoader(ds, batch_size=4, sampler=sampler))
            got = list(mine)
            assert len(mine) == len(want) == len(got)
            for (gi, gl), (wi, wl) in zip(got, want):
                assert torch.equal(gi, wi) and torch.equal(gl, wl)


@pytest.mark.parametrize("kind", ["label_shuffle", "target_noise", "uniform_gray", "gaussian"])
def test_sharded_loader_perturbations_equal_the_dataset_wrappers(kind):
    from oracle import vit_measure_ref as ref
    vt = _vt()
    g = torch.Generator().manual_seed(0)
    images, labels = torch.randn(19, 3, 4, 4, generator=g), torch.randint(0, 10, (19,), generator=g)
    mine = vt.ShardedLoader(vt.ResidentImageSet(images, labels), 5, 2, 1, shuffle=True, perturbation_type=kind,
                            epsilon=0.1, num_classes=10, noise_generator=torch.Generator().manual_seed(3))
    mine.sampler.set_epoch(9)
    want = ref.rank_loader(ref.perturbed_dataset(images, labels, kind, 0.1, 10, 42), 5, 2, 1, True, epoch=9)
    got, want = list(mine), list(want)
    assert len(got) == len(want)
    for (gi, gl), (wi, wl) in zip(got, want):
        assert torch.equal(gl, wl) and gi.shape == wi.shape and gi.dtype == wi.dtype
        if kind == "gaussian":   # fresh N(0, eps^2) noise on both sides (different generators): statistics only
            assert not torch.equal(gi, wi) and abs(float(gi.std()) - 0.1) < 0.03 and abs(float(gi.mean())) < 0.03
        else:
            assert torch.equal(gi, wi)
    with pytest.raises(ValueError):
        vt.ShardedLoader(vt.ResidentImageSet(images, labels), 5, perturbation_type="blur")


def test_resident_set_from_datasets():
    vt = _vt()
    pairs = [(torch.full((3, 2, 2), float(i)), i % 3) for i in range(5)]
    s = vt.ResidentImageSet.from_dataset(pairs, "cpu")
    assert s.images.shape == (5, 3, 2, 2) and s.labels.tolist() == [0, 1, 2, 0, 1] and len(s) == 5
    named = [(f"img{i}.jpg", torch.full((3, 2, 2), float(i))) for i in range(4)]     # THINGSInferenceDataset items
    s = vt.ResidentImageSet.from_dataset(named, "cpu")
    assert s.labels is None and s.names == [f"img{i}.jpg" for i in range(4)]
    batches = list(vt.ShardedLoader(s, 3, with_names=True))
    assert batches[0][0] == ["img0.jpg", "img1.jpg", "img2.jpg"] and batches[1][1].shape[0] == 1
    assert vt.parse_synthetic("synthetic:64:16:10") == (64, 16, 10) and vt.parse_synthetic("/data/imagenet") is None
    assert vt.parse_synthetic("synthetic") == (2048, 512, 1000)


# ------------------------------------------------------------------------------- orchestration vs the oracle
class _ScipyEvaluator:
    """hba.rsa.RSAEvaluator's interface on the host (the GPU tests use the real one)."""

    def __init__(self, rdm):
        self.rdm, self.N = np.asarray(rdm), len(rdm)

    def __call__(self, emb, want_rdm=True):
        from oracle import vit_measure_ref as ref
        rho, p = ref.rsa_tail_ref(emb.double().numpy().astype(np.float32), self.rdm)
        return rho, p, None


def _tiny_problem(seed=0, n_train=12, n_val=8, n_things=12, classes=10):
    g = torch.Generator().manual_seed(seed)
    mk = lambda n: (torch.randn(n, 3, 32, 32, generator=g), torch.randint(0, classes, (n,), generator=g))
    train, val = mk(n_train), mk(n_val)
    things = torch.randn(n_things, 3, 32, 32, generator=g)
    rdm = 1 - np.corrcoef(torch.randn(n_things, 9, generator=g).double().numpy())
    np.fill_diagonal(rdm, 0)
    return train, val, things, rdm


def _tiny_factory(classes=10):
    from oracle import vit_ref
    return lambda: vit_ref.VisionTransformerRef(img_size=32, patch_size=16, embed_dim=64, depth=1, num_heads=1,
                                                num_classes=classes)


def _write_baseline(tmp_path, factory, train, val, epochs=3, batch=4):
    """A three-epoch baseline run through the product's own epoch functions (CPU stand-in trainer): checkpoints
    + metrics CSV in the reference's formats."""
    import pandas as pd
    from hba import vit
    vt = _vt()
    torch.manual_seed(1)
    model = factory()
    tr = _TorchTrainer(model, lr=0.1)
    sched = vit.CosineAnnealingLRWithWarmup(tr, 5, 100)
    d = os.path.join(str(tmp_path), "baseline")
    tl = vt.ShardedLoader(vt.ResidentImageSet(*train), batch, shuffle=True)
    vl = vt.ShardedLoader(vt.ResidentImageSet(*val), batch)
    for epoch in range(epochs):
        tl.sampler.set_epoch(epoch)
        a = vt.train_one_epoch(tr, tl, epoch, log=None)
        sched.step()
        b, c = vt.validate(tr, vl)
        vt.save_checkpoint(epoch, model, tr, sched, a, b, c, d)
    m = pd.read_csv(os.path.join(d, "training_metrics.csv"))
    m["rsa_score"] = [0.3, 0.35, 0.4][:epochs]
    csv = os.path.join(d, "with_rsa.csv")
    m.to_csv(csv, index=False)
    return d, csv


@pytest.mark.parametrize("kind", ["uniform_gray", "label_shuffle", "target_noise"])
def test_measurement_orchestration_equals_oracle_restatement(tmp_path, monkeypatch, kind):
    from hba import vit
    from oracle import vit_measure_ref as ref
    vt = _vt()
    train, val, things, rdm = _tiny_problem()
    factory = _tiny_factory()
    ckdir, csv = _write_baseline(tmp_path, factory, train, val)
    monkeypatch.setattr(vit, "create_model", lambda name, pretrained=False, num_classes=1000: factory())
    monkeypatch.setattr(vit, "DataParallelTrainer", _TorchTrainer)
    logs = []
    got = vt.measure_perturbation_effect(
        2, kind, ckdir, csv, vt.ResidentImageSet(*train), vt.ResidentImageSet(*val), vt.ResidentImageSet(things), rdm,
        batch_size=4, num_classes=10, evaluator=_ScipyEvaluator(rdm), log=logs.append)
    ck = torch.load(os.path.join(ckdir, "checkpoint_epoch_001.pth"), weights_only=False)
    want = ref.measure_ref(ck, factory, train, val, things, rdm, 2, kind, got["baseline_loss"], 0.4, batch_size=4,
                           num_classes=10)
    assert list(got) == list(vt.RESULT_COLUMNS)
    for k in vt.RESULT_COLUMNS:
        assert got[k] == want[k], k
    assert got["baseline_rsa"] == 0.4 and got["delta_loss"] == got["perturbed_loss"] - got["baseline_loss"]
    assert any("Training perturbed epoch 2" in l for l in logs) and any("Δ loss" in l for l in logs)
    # lr of the perturbed epoch = schedule value for epoch index 1 restored from the checkpoint (0.1 * 2 / 5)
    assert ck["optimizer_state_dict"]["param_groups"][0]["lr"] == pytest.approx(0.04)


def test_measurement_skips_and_driver_csv(tmp_path, monkeypatch):
    import pandas as pd
    from hba import vit
    vt = _vt()
    train, val, things, rdm = _tiny_problem()
    factory = _tiny_factory()
    ckdir, csv = _write_baseline(tmp_path, factory, train, val)
    monkeypatch.setattr(vit, "create_model", lambda name, pretrained=False, num_classes=1000: factory())
    monkeypatch.setattr(vit, "DataParallelTrainer", _TorchTrainer)
    kw = dict(baseline_checkpoint_dir=ckdir, baseline_metrics_csv=csv, train_data=vt.ResidentImageSet(*train),
              val_data=vt.ResidentImageSet(*val), things_data=vt.ResidentImageSet(things), things_rdm=rdm, batch_size=4,
              num_classes=10, evaluator=_ScipyEvaluator(rdm), log=None)
    assert vt.measure_perturbation_effect(7, "gaussian", **kw) is None          # no baseline row (MEAS:427-430)
    os.remove(os.path.join(ckdir, "checkpoint_epoch_000.pth"))
    assert vt.measure_perturbation_effect(1, "gaussian", **kw) is None          # no checkpoint (MEAS:489-492)
    out = os.path.join(str(tmp_path), "res", "effects.csv")
    rows = vt.measure_all(out, perturb_epochs=[0, 1, 2, 7], perturbation_types=["gaussian", "target_noise"], **kw)
    assert [(r["perturb_epoch"], r["perturbation_type"]) for r in rows] == [(2, "gaussian"), (2, "target_noise")]
    df = pd.read_csv(out)
    assert list(df.columns) == list(vt.RESULT_COLUMNS) and len(df) == 2
    assert df["delta_loss"].tolist() == pytest.approx([r["delta_loss"] for r in rows], rel=1e-12)


def test_epoch_functions_equal_oracle_on_one_rank():
    from oracle import vit_measure_ref as ref
    vt = _vt()
    train, val, _, _ = _tiny_problem(seed=3)
    factory = _tiny_factory()
    torch.manual_seed(2)
    m1 = factory()
    m2 = factory()
    m2.load_state_dict(m1.state_dict())
    tr = _TorchTrainer(m1, lr=0.05)
    loader = vt.ShardedLoader(vt.ResidentImageSet(*train), 5, shuffle=True)
    loader.sampler.set_epoch(3)
    logs = []
    got = vt.train_one_epoch(tr, loader, 3, log=logs.append, log_every=2)
    opt = torch.optim.SGD(m2.parameters(), lr=0.05, momentum=0.9, weight_decay=1e-4)
    from torch.utils.data import TensorDataset
    want = ref.train_one_epoch_ref(m2, ref.rank_loader(TensorDataset(*train), 5, 1, 0, True, epoch=3), opt)
    assert got == ref.reduce_train_loss([want])
    assert len(logs) == 2 and logs[0].startswith("  [   0/3] Loss: ")
    vloss, vacc = vt.validate(tr, vt.ShardedLoader(vt.ResidentImageSet(*val), 3))
    wl, wa = ref.reduce_validation([ref.validate_rank_ref(m2, ref.rank_loader(TensorDataset(*val), 3, 1, 0, False))])
    assert (vloss, vacc) == (wl, wa)
    with pytest.raises(ValueError):
        vt.train_one_epoch(tr, [], 0)


# ------------------------------------------------------------------------------- gloo, world size 2
def _rank_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from hba import vit_train as vt
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    train, val, things, rdm = _tiny_problem(seed=4, n_val=9, n_things=12)
    torch.manual_seed(7)
    model = _tiny_factory()()
    tr = _TorchTrainer(model, lr=0.0)      # lr 0: both ranks keep identical weights without a gradient exchange
    tl = vt.ShardedLoader(vt.ResidentImageSet(*train), 4, world, rank, shuffle=True)
    tl.sampler.set_epoch(1)
    train_loss = vt.train_one_epoch(tr, tl, 1, rank, world, log=None)
    vl = vt.ShardedLoader(vt.ResidentImageSet(*val), 4, world, rank)
    val_ref = vt.validate(tr, vl, rank, world)
    val_mean = vt.validate(tr, vl, rank, world, reference_rank_sum=False)
    thl = vt.ShardedLoader(vt.ResidentImageSet(things), 8, world, rank, with_names=True)
    ev = _ScipyEvaluator(rdm)
    rsa_fixed = vt.compute_rsa_score(model, thl, rdm, rank, world, dataset_order=True, evaluator=ev)
    rsa_quirk = vt.compute_rsa_score(model, thl, rdm, rank, world, dataset_order=False, evaluator=ev)
    torch.save({"train_loss": train_loss, "val_ref": val_ref, "val_mean": val_mean, "rsa_fixed": rsa_fixed,
                "rsa_quirk": rsa_quirk}, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.destroy_process_group()


def test_collective_tails_on_gloo_world_2(tmp_path):
    import torch.multiprocessing as mp
    from torch.utils.data import TensorDataset
    from oracle import vit_measure_ref as ref
    port = 29450 + os.getpid() % 200
    mp.spawn(_rank_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (torch.load(os.path.join(str(tmp_path), f"rank{r}.pt"), weights_only=False) for r in (0, 1))
    # the oracle: per-rank values from the restated loops, combined by the restated reductions
    train, val, things, rdm = _tiny_problem(seed=4, n_val=9, n_things=12)
    torch.manual_seed(7)
    model = _tiny_factory()()
    opt = torch.optim.SGD(model.parameters(), lr=0.0, momentum=0.9, weight_decay=1e-4)
    per_rank = [ref.train_one_epoch_ref(model, ref.rank_loader(TensorDataset(*train), 4, 2, r, True, epoch=1), opt)
                for r in (0, 1)]
    assert r0["train_loss"] == r1["train_loss"] == ref.reduce_train_loss(per_rank)
    vm = [ref.validate_rank_ref(model, ref.rank_loader(TensorDataset(*val), 4, 2, r, False)) for r in (0, 1)]
    want_loss, want_acc = ref.reduce_validation(vm)
    assert r0["val_ref"] == r1["val_ref"] == (want_loss, want_acc)             # SUM of the rank means (VIT:196)
    assert r0["val_mean"][0] == want_loss / 2 and r0["val_mean"][1] == want_acc
    # RSA rows: dataset order by default = the single-rank value; reference order = its rank-major concatenation
    one_rank = ref.compute_rsa_score_ref(model, things, rdm, world_size=1)
    assert r0["rsa_fixed"][0] == pytest.approx(one_rank[0], abs=1e-12)
    assert r0["rsa_fixed"][0] == pytest.approx(ref.compute_rsa_score_ref(model, things, rdm, 2, dataset_order=True)[0], abs=1e-12)
    assert r0["rsa_quirk"][0] == pytest.approx(ref.compute_rsa_score_ref(model, things, rdm, 2, dataset_order=False)[0], abs=1e-12)
    assert abs(r0["rsa_quirk"][0] - one_rank[0]) > 1e-6                        # the interleave does change rho
    assert r1["rsa_fixed"] == (None, None) and r1["rsa_quirk"] == (None, None)  # MEAS:335-336


# ------------------------------------------------------------------------------- optimizer state (host logic)
def test_trainer_optimizer_state_layout_on_host(monkeypatch):
    """DataParallelTrainer.state_dict / load_state_dict / momentum_of: the bookkeeping between the flat
    momentum buffer (bucket order) and torch.optim.SGD's per-parameter state (model.parameters() order),
    with the SGD kernels stubbed out (their numerics are GPU-tested)."""
    from hba import ops, vit
    torch.manual_seed(0)
    model = vit.create_model("vit_tiny_test", num_classes=10)
    ps = list(model.parameters())
    # torch's own optimizer gives the layout to match
    opt = torch.optim.SGD(ps, lr=0.1, momentum=0.9, weight_decay=1e-4)
    for p in ps:
        p.grad = torch.full_like(p, 0.5)
    opt.step()
    want = opt.state_dict()

    calls = []
    monkeypatch.setattr(ops, "sgd_multi", lambda *a, **k: calls.append(("multi", a[-1])))
    monkeypatch.setattr(ops, "sgd_staged", lambda *a, **k: calls.append(("staged", a[-1])))
    tr = vit.DataParallelTrainer(model, lr=0.3, momentum=0.5, weight_decay=0.0)
    assert tr.state_dict()["state"] == {} and sorted(tr.state_dict()["param_groups"][0]) == sorted(want["param_groups"][0])
    eng = tr.eng
    eng.device, eng.precision = torch.device("cpu"), "fp32"       # host stand-in for ViTEngine._setup
    eng._ensure_grads()
    # checkpoint loaded before the first step: kept pending, handed back unchanged, applied by the first SGD call
    tr.load_state_dict(want)
    assert (tr.param_groups[0]["lr"], tr.momentum, tr.wd) == (0.1, 0.9, 1e-4) and tr._first
    back = tr.state_dict()
    assert all(torch.equal(back["state"][i]["momentum_buffer"], want["state"][i]["momentum_buffer"]) for i in want["state"])
    tr._sgd()
    assert calls == [("multi", False)]                             # momentum buffers are NOT re-initialised
    assert tr._pending_mom is None and tr._mom_valid and not tr._first
    for i, p in enumerate(ps):
        view = tr.momentum_of(p)
        assert view.shape == p.shape and torch.equal(view, want["state"][i]["momentum_buffer"])
        g = eng.grad_of[id(p)]
        assert view.data_ptr() - tr._mom.data_ptr() == g.data_ptr() - eng.flat_grad.data_ptr()
    got = tr.state_dict()
    assert sorted(got["state"]) == sorted(want["state"]) and got["param_groups"][0]["params"] == want["param_groups"][0]["params"]
    # loading into a trainer whose flat buffer exists writes through immediately and forces a host-launched step
    doubled = {"state": {i: {"momentum_buffer": v["momentum_buffer"] * 2} for i, v in want["state"].items()},
               "param_groups": [dict(want["param_groups"][0], lr=0.02)]}
    tr._graphs["stale"] = object()
    tr.load_state_dict(doubled)
    assert tr._graphs == {} and tr._first and tr._mom_valid and tr.param_groups[0]["lr"] == 0.02
    assert torch.equal(tr.momentum_of(ps[3]), want["state"][3]["momentum_buffer"] * 2)
    # a state without momentum buffers (fresh optimizer): the next step initialises them
    tr.load_state_dict({"state": {}, "param_groups": want["param_groups"]})
    tr._sgd()
    assert calls[-1] == ("multi", True) and tr.state_dict()["state"] != {}
    fresh = vit.DataParallelTrainer(vit.create_model("vit_tiny_test", num_classes=10))
    fresh.eng.device, fresh.eng.precision = torch.device("cpu"), "fp32"
    fresh.eng._ensure_grads()
    fresh._sgd()
    assert calls[-1] == ("multi", True)                            # first step of a new run: buf = grad
    with pytest.raises(ValueError):
        tr.load_state_dict({"state": {0: want["state"][0]}, "param_groups": want["param_groups"]})
    with pytest.raises(ValueError):
        bad = {i: {"momentum_buffer": torch.zeros(3)} for i in want["state"]}
        tr.load_state_dict({"state": bad, "param_groups": want["param_groups"]})


# ------------------------------------------------------------------------------- RSA over checkpoints
def _rsa_ckpt_worker(rank, world, port, ckdir, out_csv):
    import torch.distributed as dist
    from hba import vit, vit_train as vt
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    _, _, things, rdm = _tiny_problem(seed=6)
    factory = _tiny_factory()
    vit.create_model = lambda name, pretrained=False, num_classes=1000: factory()
    vt.rsa_over_checkpoints(ckdir, vt.ResidentImageSet(things), rdm, out_csv, rank=rank, world_size=world,
                            evaluator=_ScipyEvaluator(rdm), log=None)
    dist.destroy_process_group()


def test_rsa_over_checkpoints_schema_sharding_and_values(tmp_path, monkeypatch):
    """One row per checkpoint in the shipped rsa_results_final.csv schema; checkpoints sharded over a world-2
    `gloo` group give the single-process table; every rho equals the oracle's on that checkpoint's weights."""
    import pandas as pd
    import torch.multiprocessing as mp
    from hba import vit
    from oracle import vit_measure_ref as ref
    vt = _vt()
    train, val, things, rdm = _tiny_problem(seed=6)
    factory = _tiny_factory()
    ckdir, _ = _write_baseline(tmp_path, factory, train, val, epochs=3)
    monkeypatch.setattr(vit, "create_model", lambda name, pretrained=False, num_classes=1000: factory())
    out1 = os.path.join(str(tmp_path), "rsa1.csv")
    rows = vt.rsa_over_checkpoints(ckdir, vt.ResidentImageSet(things), rdm, out1, evaluator=_ScipyEvaluator(rdm), log=None)
    df = pd.read_csv(out1)
    assert list(df.columns) == ["checkpoint", "epoch", "train_loss", "val_loss", "val_acc", "rsa_score"]   # shipped schema
    assert df["checkpoint"].tolist() == [f"checkpoint_epoch_{e:03d}" for e in range(3)] and df["epoch"].tolist() == [0, 1, 2]
    metrics = pd.read_csv(os.path.join(ckdir, "training_metrics.csv"))
    assert np.allclose(df["val_loss"], metrics["val_loss"], atol=1e-6)          # the CSV keeps 6 decimals
    for r in rows:
        ck = torch.load(os.path.join(ckdir, r["checkpoint"] + ".pth"), weights_only=False)
        m = factory()
        m.load_state_dict(ck["model_state_dict"])
        assert r["rsa_score"] == ref.compute_rsa_score_ref(m, things, rdm)[0]
        assert r["val_loss"] == ck["val_loss"]
    # usable as the measurement's baseline CSV (MEAS:421-433)
    assert vt.baseline_row(out1, 2) == pytest.approx((rows[2]["val_loss"], rows[2]["rsa_score"]), rel=1e-14)
    out2 = os.path.join(str(tmp_path), "rsa2.csv")
    mp.spawn(_rsa_ckpt_worker, args=(2, 29250 + os.getpid() % 200, ckdir, out2), nprocs=2, join=True)
    assert open(out2).read() == open(out1).read()
    with pytest.raises(FileNotFoundError):
        vt.rsa_over_checkpoints(str(tmp_path / "empty"), vt.ResidentImageSet(things), rdm, evaluator=_ScipyEvaluator(rdm))


# ------------------------------------------------------------------------------- streamed ImageFolder data
def _image_tree(root, classes=3, per_class=4, val_per_class=2, size=40):
    from PIL import Image
    rng = np.random.RandomState(0)
    for split, n in (("train", per_class), ("val", val_per_class)):
        for c in range(classes):
            d = os.path.join(root, split, f"class{c}")
            os.makedirs(d)
            for i in range(n):
                Image.fromarray(rng.randint(0, 255, (size, size + 8, 3), dtype=np.uint8)).save(os.path.join(d, f"{i}.jpg"))
    return root


@pytest.mark.parametrize("kind", [None, "label_shuffle", "target_noise", "uniform_gray", "gaussian"])
def test_streamed_imagefolder_loaders_follow_the_reference_pipeline(tmp_path, kind):
    """imagenet_loaders (VIT:29-87 / MEAS:139-227) on a tiny JPEG tree: batch shapes, the label stream of a rank
    (sampler order x label perturbation) and the image perturbations; against the reference's own
    get_dataloaders where /root/reference is mounted."""
    vt = _vt()
    root = _image_tree(str(tmp_path / "data"))
    tl, vl, sampler = vt.imagenet_loaders(root, 4, 1, 2, 1, torch.device("cpu"), perturbation_type=kind, epsilon=0.1)
    assert tl.sampler is sampler
    sampler.set_epoch(3)
    got = [(x.shape, y.tolist(), float(x.abs().max()), float(x.std())) for x, y in tl]
    assert [g[0] for g in got] == [torch.Size([4, 3, 224, 224]), torch.Size([2, 3, 224, 224])]       # 12 images / 2 ranks
    if kind == "uniform_gray":
        assert all(g[2] == 0.0 for g in got)
    elif kind == "gaussian":
        assert all(abs(g[3] - 0.1) < 0.01 for g in got)
    else:
        assert all(g[2] > 1.0 for g in got)                       # normalised natural-range pixels
    vals = [(x.shape[0], y.tolist()) for x, y in vl]
    assert sum(n for n, _ in vals) == 3 and all(x.dtype == torch.float32 for x, _ in vl)   # 6 val images / 2 ranks
    if os.path.isdir("/root/reference/Training/vit_training"):
        from oracle import make_vit_measure_golden as mk
        MEAS, _ = mk.load_reference_scripts()
        rtl, rvl, rsampler = MEAS.get_dataloaders(root, 4, 1, 2, 1, perturbation_type=kind, epsilon=0.1, shuffle_seed=42)
        rsampler.set_epoch(3)
        want = [y.tolist() for _, y in rtl]
        assert [g[1] for g in got] == want
        assert [y for _, y in vals] == [y.tolist() for _, y in rvl]


def test_measurement_streams_an_imagefolder_tree(tmp_path, monkeypatch):
    """measure_perturbation_effect(train_data=None, data_path=<ImageFolder root>): the reference's real-data
    invocation (MEAS:512-517), with the device trainer replaced by the CPU stand-in."""
    from hba import vit
    from oracle import vit_ref
    vt = _vt()
    root = _image_tree(str(tmp_path / "data"))
    factory = lambda: vit_ref.VisionTransformerRef(img_size=224, patch_size=16, embed_dim=64, depth=1, num_heads=1,
                                                   num_classes=1000)
    monkeypatch.setattr(vit, "create_model", lambda name, pretrained=False, num_classes=1000: factory())
    monkeypatch.setattr(vit, "DataParallelTrainer", _TorchTrainer)
    # a one-epoch baseline on the same tree, through the same loaders
    torch.manual_seed(0)
    model = factory()
    tr = _TorchTrainer(model, lr=0.01)
    sched = vit.CosineAnnealingLRWithWarmup(tr, 5, 100)
    tl, vl, sampler = vt.imagenet_loaders(root, 4, 1, 1, 0, torch.device("cpu"))
    ckdir = str(tmp_path / "baseline")
    for epoch in range(2):
        sampler.set_epoch(epoch)
        a = vt.train_one_epoch(tr, tl, epoch, log=None)
        sched.step()
        b, c = vt.validate(tr, vl)
        vt.save_checkpoint(epoch, model, tr, sched, a, b, c, ckdir)
    g = torch.Generator().manual_seed(0)
    things = torch.randn(12, 3, 224, 224, generator=g)
    rdm = 1 - np.corrcoef(torch.randn(12, 9, generator=g).double().numpy())
    np.fill_diagonal(rdm, 0)
    csv = os.path.join(ckdir, "rsa.csv")
    vt.rsa_over_checkpoints(ckdir, vt.ResidentImageSet(things), rdm, csv, evaluator=_ScipyEvaluator(rdm), log=None)
    got = vt.measure_perturbation_effect(1, "label_shuffle", ckdir, csv, None, None, vt.ResidentImageSet(things), rdm,
                                         batch_size=4, evaluator=_ScipyEvaluator(rdm), log=None, data_path=root,
                                         num_workers=1)
    assert list(got) == list(vt.RESULT_COLUMNS) and np.isfinite(got["perturbed_loss"]) and np.isfinite(got["perturbed_rsa"])
    assert got["delta_loss"] == got["perturbed_loss"] - got["baseline_loss"]
    with pytest.raises(ValueError):
        vt.measure_perturbation_effect(1, "label_shuffle", ckdir, csv, None, None, vt.ResidentImageSet(things), rdm,
                                       evaluator=_ScipyEvaluator(rdm), log=None)


# ------------------------------------------------------------------------------- command lines of the drop-in scripts
def _script(rel):
    import importlib.util
    path = os.path.join(ROOT, "vit-project_b200", "vit_training", rel)
    spec = importlib.util.spec_from_file_location("_cli_" + os.path.basename(rel)[:-3], path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("which,rel", [("VIT", "baseline/train_vit_sgd.py"),
                                       ("MEAS", "single_epoch/measure_single_epoch_perturbation_effect.py")])
def test_script_command_lines_keep_the_reference_flags(which, rel):
    """Every flag of the reference script (read from its AST by the golden generator: VIT:247-257, MEAS:562-599)
    exists here with the same type, default and nargs; flags the reference requires stay required, except the two
    THINGS paths that `--things_csv synthetic` makes unnecessary.  Extra flags here are optional."""
    mod = _script(rel)
    actions = {a.option_strings[0]: a for a in mod.build_parser()._actions if a.option_strings and a.option_strings[0] != "-h"}
    relaxed = {"--things_img_dir", "--things_rdm_path"}
    for flag, want in GOLD["cli"][which].items():
        assert flag in actions, flag
        a = actions[flag]
        assert (a.type.__name__ if a.type else None) == want["type"], flag
        assert a.nargs == want["nargs"], flag
        if want["default"] is not None:
            assert a.default == want["default"], flag
        if flag in relaxed:
            assert want["required"] and not a.required
        else:
            assert a.required == want["required"], flag
    for flag, a in actions.items():
        if flag not in GOLD["cli"][which]:
            assert not a.required, flag
    # the reference's function names are importable from the scripts
    names = {"VIT": ("setup_distributed", "get_dataloaders", "save_checkpoint", "train_one_epoch", "validate",
                     "CosineAnnealingLRWithWarmup", "main"),
             "MEAS": ("setup_distributed", "get_dataloaders", "GaussianNoiseTransform", "UniformGrayTransform", "ShuffledLabelsDataset", "TargetNoiseDataset",
                      "THINGSInferenceDataset", "train_one_epoch", "validate", "compute_rsa_score",
                      "CosineAnnealingLRWithWarmup", "measure_perturbation_effect", "main")}[which]
    for n in names:
        assert hasattr(mod, n), n


def test_measure_script_get_dataloaders_on_cpu_tensors():
    mod = _script("single_epoch/measure_single_epoch_perturbation_effect.py")
    tl, vl, sampler = mod.get_dataloaders("synthetic:10:6:7", 4, 0, 2, 1, perturbation_type="target_noise",
                                          device=torch.device("cpu"))
    sampler.set_epoch(2)
    batches = list(tl)
    assert [x.shape[0] for x, _ in batches] == [4, 1] and len(vl) == 1 and tl.sampler is sampler
    want = torch.from_numpy(_vt().random_targets(10, 7, 42))
    order = torch.tensor(list(sampler))
    assert torch.equal(torch.cat([y for _, y in batches]), want[order])


# ------------------------------------------------------------------------------- against the reference, executed
def _start_arm(arm):
    import subprocess
    import sys
    return subprocess.Popen([sys.executable, os.path.join(ROOT, "oracle", "vit_measure_exec.py"), "--arm", arm],
                            stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, cwd=ROOT,
                            env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))


def _finish_arm(proc):
    out, err = proc.communicate(timeout=900)
    assert proc.returncode == 0, err[-3000:]
    return json.loads([l for l in out.splitlines() if l.startswith("{")][-1])


def test_host_orchestration_equals_the_reference_executed():
    """The strongest pin of SURVEY 8a row V / 8f N3: the reference's OWN `get_dataloaders`, `train_one_epoch`,
    `validate`, `save_checkpoint` (VIT) and `measure_perturbation_effect` (MEAS) are executed on the CPU
    (oracle/vit_measure_exec.py: only `timm.create_model`, `.cuda()`, `torch.load(map_location)` and the process
    group are stubbed) on a tiny JPEG tree; the product's host side with a CPU stand-in trainer, on the same files
    and RNG streams, must reproduce two baseline epochs, the metrics CSV text, and the result rows of all four
    perturbation types - bit for bit against a live reference run where /root/reference is mounted, and within
    stated tolerances of the committed output of the reference arm (tests/golden/vit_measure_exec.json) anywhere."""
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "vit_measure_exec.json")))
    assert gold["arm"] == "reference" and sorted(gold["measure"]) == sorted(_vt().PERTURBATION_TYPES)
    have_reference = os.path.isdir("/root/reference/Training/vit_training")
    procs = [_start_arm("product")] + ([_start_arm("reference")] if have_reference else [])   # side by side
    got = _finish_arm(procs[0])
    assert got["missing_epoch"] is None and gold["missing_epoch"] is None            # MEAS:427-430

    def close(a, b, tol):
        if isinstance(a, (int, str)) or a is None:
            return a == b
        return abs(a - b) <= tol * max(1.0, abs(b))

    # The committed numbers come from another run of this container image, possibly on another CPU model (other
    # BLAS kernels, last-bit differences): losses within 1e-4; a Spearman rho over 66 pairs moves in steps of
    # 4e-5 per adjacent rank swap, so near-ties may flip a few ranks: 2e-2.  The live comparison below is exact.
    LOSS, RHO = 1e-4, 2e-2

    for (a, b) in zip(got["baseline"], gold["baseline"]):
        assert all(close(x, y, LOSS) for x, y in zip(a, b)), (a, b)
    for kind, want in gold["measure"].items():
        assert list(got["measure"][kind]) == list(want) == list(_vt().RESULT_COLUMNS)
        for k in want:
            assert close(got["measure"][kind][k], want[k], RHO if "rsa" in k else LOSS), (kind, k, got["measure"][kind][k], want[k])
    # world size 2 (`gloo`): the reference's collective tails, quirks included (SURVEY C2 / C3 / C5)
    for rank in (0, 1):
        g, w = got["world2"][rank], gold["world2"][rank]
        assert close(g["train_loss"], w["train_loss"], LOSS)
        assert all(close(x, y, LOSS) for x, y in zip(g["val"], w["val"]))             # SUM over ranks of the rank means
        assert close(g["val_mean"][0], w["val"][0] / 2, LOSS)                          # ... which is twice the mean
        if rank == 0:
            assert close(g["rsa"][0], w["rsa"][0], RHO)                               # rank-interleaved rows, as the reference
            assert g["rsa_dataset_order"] == g["rsa_single_rank"]                     # default here: rows in dataset order
            assert abs(g["rsa"][0] - g["rsa_single_rank"][0]) > 1e-3                  # the interleave does change rho
        else:
            assert g["rsa"] == w["rsa"] == [None, None]                               # MEAS:335-336
    if have_reference:
        live = _finish_arm(procs[1])
        assert live["baseline"] == got["baseline"]
        assert live["metrics_csv"] == got["metrics_csv"]
        assert live["measure"] == got["measure"]                                     # every number identical
        for rank in (0, 1):
            for k in ("train_loss", "val", "rsa"):
                assert live["world2"][rank][k] == got["world2"][rank][k], (rank, k)


@pytest.mark.parametrize("n,world", [(48, 2), (48, 8), (12, 5), (7, 3), (5, 1)])
def test_rank_blocks_return_to_dataset_order_for_any_world_size(n, world):
    """`DistributedSampler(shuffle=False)` shares (padded by wrapping when W does not divide n) -> dataset order."""
    from torch.utils.data import DistributedSampler
    vt = _vt()
    emb = torch.arange(n, dtype=torch.float32).reshape(n, 1) * torch.ones(1, 3)
    blocks = [emb[list(DistributedSampler(range(n), num_replicas=world, rank=r, shuffle=False))] for r in range(world)]
    assert len({b.shape for b in blocks}) == 1
    assert torch.equal(vt.arrange_rank_blocks(blocks, True, n), emb)
    ref_order = vt.arrange_rank_blocks(blocks, False, n)                      # MEAS:333-334
    assert torch.equal(ref_order, torch.cat(blocks)[:n])
    if world > 1 and n > world:
        assert not torch.equal(ref_order, emb)
