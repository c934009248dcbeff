"""CPU tests of the analysis layer (hba.analysis, SURVEY 8f N4) against the row-by-row restatement of the
reference's notebook cells (oracle/analysis_ref.py) and the golden excerpt of the reference's own shipped
result CSVs (tests/golden/analysis.json, oracle/make_analysis_golden.py)."""
import json
import os
import subprocess
import sys

import numpy as np
import pandas as pd
import pytest

from hba import analysis, sweep
from oracle import analysis_ref as ref
from oracle import ref_loader

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "analysis.json")))
COLS = ["epoch", "test_loss", "behavioral_rsa_rho"]


def frame(rows):
    return pd.DataFrame(rows, columns=COLS)


def trimmed_baseline():
    raw = frame(GOLD["baseline_raw"])
    base = raw.loc[:raw["test_loss"].idxmin()].copy()
    assert len(base) == GOLD["baseline_trimmed_epochs"]
    return base


def test_recovery_table_matches_reference_golden():
    runs = [(name, r["start"], r["length"], frame(r["rows"])) for name, r in GOLD["length_runs"].items()]
    got = analysis.recovery_table(trimmed_baseline(), runs)
    want = pd.DataFrame(GOLD["length_expected"])
    assert list(got["run_name"]) == list(want["run_name"])
    for col in ("start_epoch", "length", "perturbation_end"):
        assert list(got[col]) == list(want[col])
    assert list(got["recovered"]) == list(want["recovered"])
    for a, b in zip(got["recovery_epoch"], want["recovery_epoch"]):
        assert (pd.isna(a) and pd.isna(b)) or int(a) == int(b)
    for a, b in zip(got["epochs_to_recovery"], want["epochs_to_recovery"]):
        assert (pd.isna(a) and pd.isna(b)) or int(a) == int(b)


def test_single_sweep_deviations_match_reference_golden():
    runs = {int(n): frame(rows) for n, rows in GOLD["single_runs"].items()}
    base = trimmed_baseline()
    for column in ("test_loss", "behavioral_rsa_rho"):
        got = analysis.deviation_at_perturbation_epoch(base, runs, column)
        want = GOLD["single_expected"][column]
        assert list(got["run"]) == [e for e, _ in want]
        assert np.allclose(got["delta_" + column].to_numpy(), [v for _, v in want], rtol=0, atol=1e-12)


@pytest.mark.parametrize("seed", range(6))
def test_vectorised_tables_equal_the_row_by_row_restatement(seed):
    """Random sweeps incl. the awkward cases: runs that never recover, runs longer than the trimmed baseline
    (fallback to the baseline minimum), missing epochs, unsorted rows, the window reaching past the run."""
    rng = np.random.default_rng(seed)
    n_base = int(rng.integers(20, 60))
    base_raw = pd.DataFrame({"epoch": np.arange(1, n_base + 1),
                             "test_loss": 100 * np.exp(-np.arange(n_base) / 15) + rng.normal(0, 1.0, n_base) + 30,
                             "behavioral_rsa_rho": rng.uniform(0.3, 0.8, n_base)})
    base = ref.trim_at_min_test_loss(base_raw)
    assert analysis.load_baseline is not None and len(base) >= 1
    runs, sruns = [], {}
    for k in range(25):
        start, length = int(rng.integers(1, 50)), int(rng.choice([1, 2, 5, 10, 20, 50]))
        n = int(rng.integers(5, 90))
        epochs = np.arange(1, n + 1)
        keep = rng.random(n) > 0.1
        loss = 30 + 100 * np.exp(-epochs / 15) + rng.normal(0, 2.0, n) + (k % 3 == 0) * 20
        df = pd.DataFrame({"epoch": epochs, "test_loss": loss, "behavioral_rsa_rho": rng.uniform(0.2, 0.8, n)})[keep]
        df = df.sample(frac=1.0, random_state=int(rng.integers(1 << 30)))          # unsorted on disk
        runs.append((f"random_target_e{start}_l{length}_{k}", start, length, df))
        sruns[int(rng.integers(1, 70))] = df
    got, want = analysis.recovery_table(base, runs), ref.recovery_table(base, runs)
    assert list(got["run_name"]) == list(want["run_name"])
    assert list(got["recovered"]) == list(want["recovered"])
    for a, b in zip(got["recovery_epoch"], want["recovery_epoch"]):
        assert (pd.isna(a) and pd.isna(b)) or int(a) == int(b)
    for column in ("test_loss", "behavioral_rsa_rho"):
        g = analysis.deviation_at_perturbation_epoch(base, sruns, column)
        w = ref.deviation_at_perturbation_epoch(base, sruns, column)
        assert list(g["run"]) == [e for e, _ in w]
        assert np.array_equal(g["delta_" + column].to_numpy(), np.array([v for _, v in w], dtype=np.float64))


def test_discovery_reads_the_layouts_the_sweep_driver_writes_and_cli_round_trip(tmp_path):
    base_cfg = {"output_base_directory": str(tmp_path / "single"), "perturb_type": "random_target"}
    rows = "epoch,train_loss,test_loss,behavioral_rsa_rho,behavioral_rsa_p_value\n"
    baseline = tmp_path / "baseline.csv"
    baseline.write_text(rows + "".join(f"{e},{100 - e},{90 - 2 * e},{0.4 + 0.01 * e},0.0\n" for e in range(1, 11)))
    for e in (2, 5):
        cfg = sweep.condition_config(base_cfg, {"training_run": e, "perturb_length": 1}, "sweep")
        with open(cfg["training_res_path"], "w") as f:
            f.write(rows + "".join(f"{k},{100 - k},{91 - 2 * k + (3 if k == e else 0)},{0.39 + 0.01 * k},0.0\n" for k in range(1, 11)))
    len_cfg = {"output_base_directory": str(tmp_path / "length"), "perturb_type": "random_target"}
    for e, l in ((2, 2), (3, 5)):
        cfg = sweep.condition_config(len_cfg, {"training_run": e, "perturb_length": l}, "length")
        with open(cfg["training_res_path"], "w") as f:
            f.write(rows + "".join(f"{k},{100 - k},{(200 if e <= k < e + l else 90 - 2 * k + (5 if k < e + l + 2 else 0))},0.5,0.0\n"
                                   for k in range(1, 11)))
    runs = analysis.discover_single_sweep(str(tmp_path / "single"))
    assert sorted(runs) == [2, 5]
    s = analysis.single_sweep_summary(str(baseline), str(tmp_path / "single"))
    assert list(s["run"]) == [2, 5] and np.allclose(s["delta_test_loss"], [4.0, 4.0]) and np.allclose(s["delta_behavioral_rsa_rho"], -0.01)
    lr = analysis.discover_length_runs(str(tmp_path / "length"))
    assert [(n, a, b) for n, a, b, _ in lr] == [("random_target_e2_l2", 2, 2), ("random_target_e3_l5", 3, 5)]
    t = analysis.length_grid_summary(str(baseline), str(tmp_path / "length"))
    assert list(t["perturbation_end"]) == [3, 7] and list(t["recovery_epoch"]) == [6, 10] and list(t["epochs_to_recovery"]) == [3, 3]
    out = tmp_path / "recovery.csv"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "analyze_sweep.py"), "--kind", "length", "--baseline",
                        str(baseline), "--sweep-dir", str(tmp_path / "length"), "--out", str(out)],
                       capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    back = pd.read_csv(out)
    assert list(back["recovery_epoch"]) == [6, 10] and list(back["recovered"]) == [True, True]


@pytest.mark.skipif(not os.path.isdir("/root/reference/Data/clip_results"), reason="reference data not mounted")
def test_full_reference_result_set_summary():
    """All shipped conditions through the product functions: counts and checksums of the golden generator."""
    data = "/root/reference/Data/clip_results"
    base_csv = os.path.join(data, "baseline_clip_results_seed1.csv")
    t = analysis.length_grid_summary(base_csv, os.path.join(data, "perturb_length_experiments_baselineseed1_perturbseed0"))
    s = analysis.single_sweep_summary(base_csv, os.path.join(data, "single_sweep_experiments"))
    f = GOLD["full_summary"]
    assert len(t) == f["n_length_runs"] and int(t["recovered"].sum()) == f["n_recovered"]
    assert int(t["epochs_to_recovery"].dropna().sum()) == f["sum_epochs_to_recovery"]
    assert len(s) == f["n_single_with_deviation"]
    assert abs(float(s["delta_test_loss"].sum()) - f["sum_delta_test_loss"]) < 1e-9
    assert abs(float(s["delta_behavioral_rsa_rho"].sum()) - f["sum_delta_rsa"]) < 1e-9


# ------------------------------------------------------------------------------- FIG2
def _fig2_runs():
    return {name: {int(e): frame(rows) for e, rows in runs.items()} for name, runs in GOLD["fig2_runs"].items()}


def test_perturbation_type_comparison_matches_reference_golden():
    """FIG2 cells 5-9 on the excerpt of the reference's shipped Data/clip_results/{image_noise, uniform_target,
    label_shuffle, target_noise}: the deltas the notebook plots, and the row-by-row restatement."""
    base = trimmed_baseline()
    runs = _fig2_runs()
    got = analysis.perturbation_type_comparison(base, runs)
    assert list(analysis.FIG2_TARGET_EPOCHS) == GOLD["fig2_target_epochs"] == ref.FIG2_TARGET_EPOCHS
    assert list(got.columns) == ["perturbation", "epoch", "delta_test_loss", "delta_behavioral_rsa_rho"]
    assert len(got) == 4 * 7 and list(got["perturbation"].unique()) == ["image_noise", "blank_image", "label_shuffle", "target_noise"]
    again = ref.fig2_type_deviations(base, runs)
    for name, want in GOLD["fig2_expected"].items():
        sub = got[got["perturbation"] == name]
        assert list(sub["epoch"]) == GOLD["fig2_target_epochs"]
        for col, key in (("delta_test_loss", "test_loss"), ("delta_behavioral_rsa_rho", "behavioral_rsa_rho")):
            w = np.array([np.nan if v is None else v for v in want[key]])
            assert np.array_equal(sub[col].to_numpy(), w, equal_nan=True)
            assert np.array_equal(np.array(again[name][key]), w, equal_nan=True)
    # the qualitative finding of the figure: every perturbation hurts more the later it comes
    ls = got[got["perturbation"] == "label_shuffle"]["delta_test_loss"].to_numpy()
    assert (np.diff(ls) > 0).all()


def test_perturbation_type_comparison_missing_pieces(tmp_path):
    base = pd.DataFrame({"epoch": [1, 2, 3], "test_loss": [9.0, 8.0, 7.0], "behavioral_rsa_rho": [0.1, 0.2, 0.3]})
    run2 = pd.DataFrame({"epoch": [1, 2, 3], "test_loss": [9.0, 8.5, 7.0], "behavioral_rsa_rho": [0.1, 0.15, 0.3]})
    run3_no_row = pd.DataFrame({"epoch": [1, 2], "test_loss": [9.0, 8.0], "behavioral_rsa_rho": [0.1, 0.2]})
    runs = {"a": {2: run2, 3: run3_no_row, 5: run2}, "b": {}}
    got = analysis.perturbation_type_comparison(base, runs, target_epochs=(2, 3, 5))
    want = ref.fig2_type_deviations(base, runs, target_epochs=[2, 3, 5])
    a = got[got["perturbation"] == "a"]
    assert a["delta_test_loss"].tolist()[0] == 0.5 and np.isnan(a["delta_test_loss"].tolist()[1:]).all()
    assert abs(a["delta_behavioral_rsa_rho"].tolist()[0] + 0.05) < 1e-15
    assert got[got["perturbation"] == "b"][["delta_test_loss", "delta_behavioral_rsa_rho"]].isna().all().all()
    for name in ("a", "b"):
        sub = got[got["perturbation"] == name]
        assert np.array_equal(sub["delta_test_loss"].to_numpy(), np.array(want[name]["test_loss"]), equal_nan=True)
        assert np.array_equal(sub["delta_behavioral_rsa_rho"].to_numpy(), np.array(want[name]["behavioral_rsa_rho"]), equal_nan=True)
    # directory form + CLI
    root = tmp_path / "results"
    for d in ("label_shuffle", "image_noise"):
        (root / d).mkdir(parents=True)
        run2.to_csv(root / d / "training_res_run2.csv", index=False)
    (root / "label_shuffle" / "notes.txt").write_text("x")
    bcsv = tmp_path / "baseline.csv"
    pd.concat([base, pd.DataFrame({"epoch": [4], "test_loss": [7.5], "behavioral_rsa_rho": [0.3]})]).to_csv(bcsv, index=False)
    t = analysis.perturbation_type_summary(str(bcsv), str(root), target_epochs=(2,))
    by = dict(zip(t["perturbation"], t["delta_test_loss"]))
    assert by["label_shuffle"] == 0.5 and by["image_noise"] == 0.5 and np.isnan(by["blank_image"]) and np.isnan(by["target_noise"])


def test_vit_summary_table_reproduces_the_shipped_csv(tmp_path):
    """Data/vit_results/perturbation_effects.csv -> perturbation_summary_table.csv, text for text."""
    eff = pd.DataFrame(GOLD["vit_effects_rows"])
    got = analysis.vit_perturbation_summary(eff)
    assert got.to_csv(index=False) == GOLD["vit_summary_csv"]
    assert got.to_dict("records") == ref.vit_summary_table(eff)
    src = tmp_path / "effects.csv"
    eff.to_csv(src, index=False)
    out = tmp_path / "summary.csv"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "analyze_sweep.py"), "--kind", "vit-summary", "--effects",
                        str(src), "--out", str(out)], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert out.read_text() == GOLD["vit_summary_csv"]
    # the columns are the ones hba.vit_train writes
    from hba import vit_train
    assert set(analysis.VIT_SUMMARY_COLUMNS) <= set(vit_train.RESULT_COLUMNS)


def _excerpt_tree(root):
    """The golden excerpt laid out like the reference's Data/ tree: the baseline CSV, the FIG2 runs as
    clip_results/<type dir>/training_res_run{e}.csv, and Data/vit_results' two CSVs."""
    clip = root / "clip_results"
    clip.mkdir(parents=True)
    frame(GOLD["baseline_raw"]).to_csv(clip / "baseline_clip_results_seed1.csv", index=False)
    for name, runs in GOLD["fig2_runs"].items():
        d = clip / analysis.FIG2_TYPE_DIRS[name]
        d.mkdir()
        for e, rows in runs.items():
            frame(rows).to_csv(d / f"training_res_run{e}.csv", index=False)
    vit = root / "vit_results"
    vit.mkdir()
    pd.DataFrame(GOLD["vit_effects_rows"]).to_csv(vit / "perturbation_effects.csv", index=False)
    (vit / "perturbation_summary_table.csv").write_text(GOLD["vit_summary_csv"])
    return str(root)


def test_fig2_tables_from_the_reference_tree_directly(tmp_path):
    """The directory-level entry points on the reference's own Data/ tree where it is present, else on the golden
    excerpt of it laid out the same way; the expected values are the reference's either way."""
    data = os.path.join(ref_loader.REFERENCE_ROOT, "Data")
    if not os.path.isdir(os.path.join(data, "clip_results")):
        data = _excerpt_tree(tmp_path / "Data")
    t = analysis.perturbation_type_summary(os.path.join(data, "clip_results", "baseline_clip_results_seed1.csv"),
                                           os.path.join(data, "clip_results"))
    for name, want in GOLD["fig2_expected"].items():
        sub = t[t["perturbation"] == name]
        assert np.array_equal(sub["delta_test_loss"].to_numpy(), np.array(want["test_loss"], dtype=np.float64), equal_nan=True)
        assert np.array_equal(sub["delta_behavioral_rsa_rho"].to_numpy(),
                              np.array(want["behavioral_rsa_rho"], dtype=np.float64), equal_nan=True)
    out = tmp_path / "fig2.csv"
    p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "analyze_sweep.py"), "--kind", "types", "--baseline",
                        os.path.join(data, "clip_results", "baseline_clip_results_seed1.csv"), "--sweep-dir",
                        os.path.join(data, "clip_results"), "--out", str(out)], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0, p.stderr
    assert len(pd.read_csv(out)) == 28
    shipped = open(os.path.join(data, "vit_results", "perturbation_summary_table.csv")).read()
    assert analysis.vit_perturbation_summary(os.path.join(data, "vit_results", "perturbation_effects.csv")).to_csv(index=False) == shipped


# ------------------------------------------------------------------------------- the notebooks, executed
@pytest.mark.skipif(not os.path.isdir("/root/reference/Figures"), reason="reference not mounted")
def test_analysis_layer_equals_the_notebooks_executed():
    """The reference's figure notebooks (fig2 / fig3 / fig4) are executed cell by cell on the reference's own Data/
    tree (oracle/run_notebook.py: plotting libraries mocked, nothing else touched); the tables they compute are
    compared with the analysis layer's directory-level entry points: all 136 length-grid runs, all 98
    single-epoch runs, 4 x 7 perturbation-type deltas."""
    from oracle import run_notebook as rn
    data = "/root/reference/Data/clip_results"
    base_csv = os.path.join(data, "baseline_clip_results_seed1.csv")
    # fig2 (cells 3-7)
    ns = rn.run_cells("fig2", stop_after=7)
    t = analysis.perturbation_type_summary(base_csv, data)
    for name, loss_var, ba_var in (("image_noise", "in_dev", "in_ba"), ("blank_image", "bi_dev", "bi_ba"),
                                   ("label_shuffle", "ls_dev", "ls_ba"), ("target_noise", "tn_dev", "tn_ba")):
        sub = t[t["perturbation"] == name]
        assert list(sub["epoch"]) == list(ns["target_epochs"])
        assert np.array_equal(sub["delta_test_loss"].to_numpy(), np.array(ns[loss_var], dtype=np.float64), equal_nan=True)
        assert np.array_equal(sub["delta_behavioral_rsa_rho"].to_numpy(), np.array(ns[ba_var], dtype=np.float64), equal_nan=True)
    # fig3 (cells 4-10)
    ns = rn.run_cells("fig3", stop_after=10)
    s = analysis.single_sweep_summary(base_csv, os.path.join(data, "single_sweep_experiments"))
    want_loss = dict(zip(ns["run_numbers_deviation"], ns["perturbation_deviations"]))
    want_ba = dict(zip(ns["run_numbers_deviation_ba"], ns["perturbation_deviations_ba"]))
    assert len(want_loss) == 98 and sorted(want_loss) == list(s["run"])
    assert [want_loss[r] for r in s["run"]] == list(s["delta_test_loss"])
    assert [want_ba[r] for r in s["run"]] == list(s["delta_behavioral_rsa_rho"])
    # fig4 (cells 4-12)
    ns = rn.run_cells("fig4", stop_after=12)
    g = analysis.length_grid_summary(base_csv, os.path.join(data, "perturb_length_experiments_baselineseed1_perturbseed0"))
    want = {r["run_name"]: r for r in ns["recovery_data"]}
    assert len(want) == 136 and sorted(want) == sorted(g["run_name"])
    for row in g.to_dict("records"):
        w = want[row["run_name"]]
        assert (row["start_epoch"], row["length"], row["perturbation_end"]) == (w["start_epoch"], w["length"], w["perturbation_end"])
        assert bool(row["recovered"]) == bool(w["recovered"])
        if w["recovered"]:
            assert int(row["recovery_epoch"]) == w["recovery_epoch"] and int(row["epochs_to_recovery"]) == w["epochs_to_recovery"]
        else:
            assert pd.isna(row["recovery_epoch"]) and pd.isna(row["epochs_to_recovery"])
