#!/usr/bin/env python
"""bench.py — CLIP-HBA-Behavior training throughput (images/s) on N B200s.

Workload (BASELINE.json configs[0], the configuration `metric` is quoted on): ViT-L/14 CLIP +
DoRA (rank 32) on the last 2 vision blocks and the last text block, batch 32 synthetic 224^2 images
-> random 66-D targets, MSE, AdamW(lr 3e-4).  One "step" = one full training step exactly as the
reference does it per batch (NEW:985-1003): the whole vision trunk AND the text tower are recomputed
every step (no activation cache inside the timed region), forward + live-sub-graph backward + DoRA
backward + optimiser step.  N > 1 runs N independent replicas (one sweep condition per GPU — the
path shards as independent runs, SURVEY §8e): weak scaling, no data-path collective.

  value : images/s with inputs resident in HBM (device-timed, max over ranks)
  e2e   : same metric through the public API (functions.*: CLIPHBA + DoRALayer + FusedAdamW) with
          pinned HOST images/targets copied in and the loss read back every step
  roofline : the tcgen05 GEMM kernel, algorithmic FLOPs / CUDA-event time of its launches over a >= 2 s
          host-launched pass, against MEASURED_PEAKS.json: the burst figure when the pass kept the SM clock near
          its maximum, the sustained one otherwise (both fractions are in the line)
  fp32_mode / roofline_hbm / sweep / vit_b16 : the parity mode on the same workload, the HBM-bound kernels
          against the measured HBM peak, a scheduler-run slice of the 136-condition grid, ViT-B/16 data parallel
  cpu_baseline : the oracle port (oracle/clip_ref.py + oracle/dora_ref.py, PyTorch fp32 on the host
          cores) on a bounded sample of the same workload

`--impl reference` times that CPU implementation as the reference arm.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
T_START = time.perf_counter()   # process start, for --time-budget
SWEEP_RESERVE_S = 150.0         # kept back from the budget for what follows the sweep slice (ViT section, CPU arm, teardown)
SWEEP_MIN_S = 30.0              # ... but the slice always gets this much
for _p in (ROOT, os.path.join(ROOT, "vit-project_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "CLIP-HBA train imgs/s"
UNIT = "images/s"
N_CLASSES = 66


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps of the headline and e2e regions (the fp32-mode and ViT-B/16 sections time "
                         "max(3, min(steps, 10)) steps and report that count as their 'steps')")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--backbone", default="ViT-L/14")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-sample-images", type=int, default=0,
                    help="images per CPU-arm step (0 = the stated batch: same config as the GPU arm)")
    ap.add_argument("--sweep-per-gpu", type=int, default=4, help="grid conditions per GPU in the scheduler-run slice")
    ap.add_argument("--sweep-timeout", type=float, default=300.0, help="limit of the scheduler-run sweep slice [s]")
    ap.add_argument("--time-budget", type=float, default=700.0,
                    help="wall clock the whole run should stay within [s]: the scheduler-run sweep slice (the one section "
                         "whose duration depends on the host: process start-up of N workers) gets what is left of it "
                         "minus a reserve for the ViT section and the teardown, at most --sweep-timeout")
    ap.add_argument("--no-fp32", action="store_true")
    ap.add_argument("--no-hbm-kernels", action="store_true")
    ap.add_argument("--roofline-seconds", type=float, default=2.6,
                    help="minimum duration of the event-bracketed GEMM roofline pass")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--no-vit", action="store_true")
    ap.add_argument("--sweep-only", action="store_true", help="debug: measure only the sweep section")
    ap.add_argument("--vit-batch", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last of them computed (loss, trainable parameters "
                         "after the optimiser step, their gradients) to DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, n):
    return {"workload": f"CLIP-HBA-Behavior {args.backbone} + DoRA r32 (last 2 vision + 1 text out_proj), "
                        f"batch {args.batch}/GPU, 224x224 synthetic images -> random 66-D targets, MSE, "
                        "AdamW lr 3e-4; full trunk + text tower recomputed every step (no activation cache)",
            "global_batch": args.batch * n, "parallelism": f"{n} independent replicas (one condition per GPU)",
            "l2": "per-step working set (>= 1.3 GB of activations and 0.8 GB of weights) exceeds the "
                  "126 MB L2; no explicit flush",
            "precision_mode": args.precision}


# ----------------------------------------------------------------------------- CPU reference arm
def build_cpu_reference(backbone, rank=32):
    import torch
    from oracle import clip_ref, dora_ref
    from functions.spose_dimensions import classnames66
    sd = clip_ref.synthetic_state_dict(backbone, seed=1)
    tokens = torch.stack([clip_ref.tokenize(c) for c in classnames66])
    model = dora_ref.CLIPHBARef(clip_ref.build_model(sd), tokens)
    torch.manual_seed(123)
    dora_ref.apply_dora_ref(model, 2, 1, r=rank)
    dora_ref.switch_dora_ref(model)
    return model


def cpu_step_fn(model, n_images):
    import torch
    g = torch.Generator().manual_seed(0)
    images = torch.randn(n_images, 3, 224, 224, generator=g)
    targets = torch.randn(n_images, N_CLASSES, generator=g) * 9.5 + 5.75
    opt = torch.optim.AdamW(model.parameters(), lr=3e-4)
    crit = torch.nn.MSELoss()

    def step():
        opt.zero_grad()
        loss = crit(model(images), targets)
        loss.backward()
        opt.step()
        return float(loss)
    return step


def eager_gpu_baseline(args, device):
    import torch
    model = build_cpu_reference(args.backbone).to(device)
    g = torch.Generator().manual_seed(0)
    images = torch.randn(args.batch, 3, 224, 224, generator=g).to(device)
    targets = (torch.randn(args.batch, N_CLASSES, generator=g) * 9.5 + 5.75).to(device)
    opt = torch.optim.AdamW([p for p in model.parameters() if p.requires_grad], lr=3e-4)
    crit = torch.nn.MSELoss()
    res = {}
    for tag, ctx in (("fp32", None), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        def step():
            opt.zero_grad()
            if ctx is None:
                loss = crit(model(images), targets)
            else:
                with ctx:
                    loss = crit(model(images).float(), targets)
            loss.backward()
            opt.step()
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        e0.record()
        for _ in range(reps):
            step()
        e1.record()
        torch.cuda.synchronize()
        res[tag] = {"value": args.batch * reps / (e0.elapsed_time(e1) / 1e3), "unit": UNIT,
                    "ms_per_step": e0.elapsed_time(e1) / reps}
    res["what"] = (f"oracle port (oracle/clip_ref.py + dora_ref.py) on cuda, batch {args.batch}, fwd+bwd+AdamW, "
                   "text tower recomputed; torch eager, allow_tf32 off")
    del model, opt
    torch.cuda.empty_cache()
    return res


def run_reference(args):
    """The reference's CPU path (restated: oracle port) on all host cores; one step = a bounded
    sample of `cpu_sample_images` images of the same workload."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    n_img = args.cpu_sample_images or args.batch
    model = build_cpu_reference(args.backbone)
    step = cpu_step_fn(model, n_img)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        loss = step()
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, loss, model)
    value = n_img * args.steps / dt
    sample = (f"{n_img} images per step = the stated batch (fwd + bwd + AdamW, text tower recomputed each "
              f"step), {args.steps} steps, PyTorch fp32, {torch.get_num_threads()} threads; oracle port "
              "(the reference is pure Python on an un-vendored CLIP: there is no reference binary to build)")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args, args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample, "sample_batch": n_img},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:   # make sure the poller is gone: a live `nvidia-smi -lms` slows every later CUDA call
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            self.proc.wait()
        sm, mx, reasons = [], [], set()
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                  "sw_power_cap"), parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------- B200 arm
def build_gpu_model(args, device):
    """The public API a user of the reference calls: CLIPHBA + apply_dora_to_ViT + switch_dora_layers
    (NEW:1133-1152) from the drop-in functions module, AdamW via its make_optimizer."""
    import torch
    import functions._pipeline_core as core
    from functions.spose_dimensions import classnames66
    os.environ.setdefault("HBA_SYNTHETIC_OK", "1")
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        model = core.CLIPHBA(classnames66, backbone_name=args.backbone, pos_embedding=True)
    torch.manual_seed(123)
    core.apply_dora_to_ViT(model, n_vision_layers=2, n_transformer_layers=1, r=32)
    core.switch_dora_layers(model, freeze_all=True, dora_state=True)
    model.to(device)
    model.train()
    opt = core.make_optimizer(model, 3e-4)
    return model, opt


def dump_outputs(out_dir, loss, model):
    """What a caller of the timed step holds after its last call: the loss, the trainable (DoRA) parameters after
    the optimiser step and the gradients that step applied.  Inputs and initial weights are seeded, so two builds
    run with the same arguments can be compared file by file (DoRA r32 on 2 + 1 blocks of ViT-L/14: 1.5 MB)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": torch.as_tensor(loss)}
    for name, p in model.named_parameters():
        if p.requires_grad:
            arrays[f"param.{name}"] = p
            if p.grad is not None:
                arrays[f"grad.{name}"] = p.grad
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


EPOCHS_PER_CONDITION = 55  # reference sweep mean: 64.0 h * 3600 / 97 conditions / 43.5 s per epoch


def measure_sweep(args, device, world):
    """Perturbation-sweep throughput (BASELINE.json metric, second half): epochs of the drop-in
    `train_model` (NEW:782-1063: 1444 train + 362 test + 48 RSA images, per-epoch eval, RSA, CSV row,
    DoRA + random-state checkpoints) on HBM-resident synthetic data with the frozen-trunk cache.
    One condition = EPOCHS_PER_CONDITION epochs; one condition per GPU, no collective."""
    import tempfile
    import numpy as np
    import scipy.io
    import torch
    import functions.new_cvpr_train_behavior_things_pipeline as NEW
    from functions import _pipeline_core as core
    from hba.data import ResidentLoader, ResidentStore
    n_train, n_test, n_rsa, bs = 1444, 362, 48, args.batch
    g = torch.Generator(device=device).manual_seed(5)
    imgs = torch.randn(n_train + n_test, 3, 224, 224, device=device, generator=g)
    tgts = torch.randn(n_train + n_test, N_CLASSES, device=device, generator=g) * 9.5 + 5.75
    rsa_imgs = torch.randn(n_rsa, 3, 224, 224, device=device, generator=g)
    store = ResidentStore(None, device, names=[f"img{i}" for i in range(n_train + n_test)], images=imgs,
                          targets=tgts)
    rstore = ResidentStore(None, device, names=[f"rsa{i}" for i in range(n_rsa)], images=rsa_imgs)
    tmp = tempfile.mkdtemp(prefix="hba_sweep_")
    rdm = 1 - np.corrcoef(np.random.default_rng(2).standard_normal((n_rsa, 66)))
    np.fill_diagonal(rdm, 0)
    scipy.io.savemat(os.path.join(tmp, "RDM48_triplet.mat"), {"RDM48_triplet": rdm})

    class _Rsa:  # carries the attributes behavioral_RSA reads from loader.dataset (NEW:636)
        RDM48_triplet_dir = os.path.join(tmp, "RDM48_triplet.mat")

        def __len__(self):
            return n_rsa

    model, opt = build_gpu_model(args, device)
    # (the frozen CLIP and its engine are shared per process, functions._pipeline_core.load_clip_to_cpu:
    # undo the headline measurement's "recompute the text tower every step" switch - the pipeline's own
    # default caches the constant text trunk, NEW:282)
    model.clip_model.hba_engine().cache_text = True
    core.enable_trunk_cache(model, n_train + n_test + n_rsa)
    gen = torch.Generator()
    gen.manual_seed(1)
    perm = torch.randperm(n_train + n_test, generator=torch.Generator().manual_seed(1)).tolist()
    tl = ResidentLoader(store, bs, shuffle=True, generator=gen, index_map=perm[:n_train])
    el = ResidentLoader(store, bs, shuffle=False, index_map=perm[n_train:])
    rl = ResidentLoader(rstore, bs, shuffle=False, dataset=_Rsa())
    crit = torch.nn.MSELoss()
    import logging
    logging.disable(logging.CRITICAL)

    def run(first, last, tag):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
            NEW.train_model(model, tl, el, rl, device, opt, crit, epochs=last,
                            training_res_path=os.path.join(tmp, "res.csv"), training_run=2, perturb_length=1,
                            perturb_seed=42, mean=5.75, std=9.5, perturb_distribution="target",
                            perturb_type="random_target", logger=None, early_stopping_patience=1000,
                            dora_parameters_path=os.path.join(tmp, "dora"),
                            random_state_path=os.path.join(tmp, "rand"), dataloader_generator=gen,
                            resume_from_epoch=first,
                            previous_training_res_path=os.path.join(tmp, "res.csv") if first else None)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    k = 6
    t_fill = run(0, 1, "fill")          # epoch 1: trunk computed once per image, cache filled
    t_capture = run(1, 2, "capture")    # epoch 2: first cached epoch, the step / forward graphs are captured
    t_cached = run(2, 2 + k, "cached")  # epochs 3..k+2: steady state of a 55-epoch condition
    logging.disable(logging.NOTSET)
    sec_epoch = t_cached / k
    imgs_epoch = n_train + n_test + n_rsa
    sec_cond = t_fill + t_capture + (EPOCHS_PER_CONDITION - 2) * sec_epoch
    return {"conditions_per_hour": world * 3600.0 / sec_cond, "unit": "conditions/h",
            "epochs_per_condition": EPOCHS_PER_CONDITION, "sec_per_epoch_cached": sec_epoch,
            "sec_first_epoch_cache_fill": t_fill, "sec_second_epoch_graph_capture": t_capture,
            "sec_per_condition": sec_cond,
            "images_per_epoch": imgs_epoch,
            "blended_images_per_s": world * imgs_epoch / sec_epoch,
            "config": "train_model epochs on 1444/362/48 synthetic HBM-resident images, batch %d, random_target "
                      "window, per-epoch eval + RSA + CSV + DoRA/random-state checkpoints, frozen-trunk cache, CUDA-graph "
                      "cached steps; wall clock incl. host; one condition = cache-fill epoch + capture epoch + 53 "
                      "steady-state epochs" % bs,
            "reference_baseline": "1.52 conditions/h, 43.5 s/epoch on one unnamed GPU (BASELINE.md, derived)"}


def measure_sweep_scheduler(args, world, rank, dist):
    """BASELINE.json configs[3] (the variable-length perturbation grid) through the scheduler: rank 0 runs
    tools/grid_sweep_bench.py (hba.sweep.run_sweep over GPUs 0..world-1, `--sweep-per-gpu` grid conditions per GPU
    taken longest-first from the conditions that start at epoch <= 10: weak scaling) while the other ranks
    wait on the rendezvous store, their GPUs idle.  conditions/hour = conditions / wall clock from the first
    worker spawn to the last result (worker start-up, cache fill, graph capture and every file included)."""
    import tempfile
    from datetime import timedelta
    key = "hba_sweep_slice_done"
    store = None
    if dist is not None:
        from torch.distributed import distributed_c10d
        store = distributed_c10d._get_default_store()
        dist.barrier()
    if rank != 0:
        store.wait([key], timedelta(seconds=1800))   # CPU-side wait: no NCCL kernel spins on this GPU meanwhile
        return None
    res = {}
    try:
        out_path = os.path.join(tempfile.mkdtemp(prefix="hba_sched_"), "slice.json")
        env = {k: v for k, v in os.environ.items()
               if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "GROUP_RANK",
                            "ROLE_RANK", "LOCAL_WORLD_SIZE", "ROLE_WORLD_SIZE", "TORCHELASTIC_RUN_ID",
                            "HBA_STEP_GRAPH", "HBA_TEXT_STREAM")}
        cmd = [sys.executable, os.path.join(ROOT, "tools", "grid_sweep_bench.py"), "--kind", "grid",
               "--gpus", ",".join(str(i) for i in range(world)), "--per-gpu", str(args.sweep_per_gpu),
               "--max-start", "10", "--batch-size", str(args.batch), "--backbone", args.backbone,
               "--root", tempfile.mkdtemp(prefix="hba_grid_"), "--out", out_path]
        t0 = time.perf_counter()
        # the slice may use what is left of the run's time budget (minus a reserve for the ViT section and the
        # teardown): a driver that limits the whole run must still get its JSON line, which is printed at the end
        limit = float(args.sweep_timeout)
        budget = getattr(args, "time_budget", None)
        if budget:
            limit = max(SWEEP_MIN_S, min(limit, budget - (t0 - T_START) - SWEEP_RESERVE_S))
        # own session: on a timeout the tool AND the worker processes it spawned are killed together, so that no
        # stray worker holds a GPU when the next section starts
        proc = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                start_new_session=True)
        try:
            out_txt, err_txt = proc.communicate(timeout=limit)
        except subprocess.TimeoutExpired:
            import signal
            os.killpg(proc.pid, signal.SIGKILL)
            out_txt, err_txt = proc.communicate()
            err_txt = f"timed out after {limit:.1f} s\n" + (err_txt or "")
        proc.stdout_text, proc.stderr_text = out_txt, err_txt
        if os.path.exists(out_path):
            full = json.load(open(out_path))
            res = {k: v for k, v in full.items() if k != "per_condition"}
            res["unit"] = "conditions/h"
            res["epochs_per_condition"] = [c["epochs_trained"] for c in full["per_condition"]]
            res["tool_wall_s"] = time.perf_counter() - t0
        if proc.returncode != 0:
            res["error"] = (proc.stderr_text or proc.stdout_text or "")[-400:]
    except Exception as exc:
        res["error"] = f"{type(exc).__name__}: {exc}"[:300]
    if store is not None:
        store.set(key, "1")
    return res


def measure_vit(args, device, world, dist):
    """BASELINE.json configs[2]: ViT-B/16 classification training, data parallel (VIT = Training/
    vit_training/baseline/train_vit_sgd.py): batch 256 per GPU, synthetic 224^2 images / 1000 classes,
    SGD 0.1 / 0.9 / 1e-4, bf16 tensor-core GEMMs, one NCCL all-reduce per block bucket overlapped with
    the backward pass, CUDA-graph step.  Whole-job images/s, device-timed, max over ranks."""
    import torch
    from hba import ops, vit
    rank = int(os.environ.get("RANK", "0"))
    torch.manual_seed(0)
    model = vit.create_model("vit_base_patch16_224", num_classes=1000).to(device)
    tr = vit.DataParallelTrainer(model, lr=0.1, momentum=0.9, weight_decay=1e-4, use_graph=True)
    tr.broadcast_parameters()
    batch = args.vit_batch
    g = torch.Generator(device=device).manual_seed(rank)
    images = torch.randn(batch, 3, 224, 224, device=device, generator=g)
    labels = torch.randint(0, 1000, (batch,), device=device, generator=g)
    for _ in range(3):
        loss, _ = tr.step(images, labels)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    steps = max(3, min(args.steps, 10))
    c0 = ops.COUNTERS["launches"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, _ = tr.step(images, labels)
    e1.record()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    value = world * batch * steps / (ms / 1e3)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = json.load(open(peaks_path))["bf16_tflops_sustained"] if os.path.exists(peaks_path) else 1400.0
    tflops = value / world * 105.3e9 / 1e12   # SURVEY 8d: 3 x 35.1 GFLOP per image
    loss_val, n_launch = float(loss), ops.COUNTERS["launches"] - c0
    exposed = None
    if dist is not None and world > 1:
        # the same step with the gradient all-reduces left out (the ranks then drift apart - nothing is measured
        # after this): what the collectives cost beyond what the backward pass hides
        try:
            tr.reducer.enabled = False
            tr._graphs.clear()
            # (rank-local on purpose: no collective inside this block, so a failure on one rank cannot strand the others)
            for _ in range(3):
                tr.step(images, labels)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(steps):
                tr.step(images, labels)
            f1.record()
            torch.cuda.synchronize()
            ms_local = f0.elapsed_time(f1)
            exposed = {"ms_per_step_without_allreduce": ms_local / steps,
                       "exposed_collective_ms_per_step": (ms - ms_local) / steps,
                       "what": "same captured step with the bucket all-reduces left out, timed on this rank"}
        except Exception as exc:   # reporting only
            exposed = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        finally:
            tr.reducer.enabled = True
    try:   # (never let the teardown cost the numbers above)
        tr.close()
    except Exception as exc:
        exposed = dict(exposed or {}, close_error=f"{type(exc).__name__}: {exc}"[:200])
    del tr, model
    return {"metric": "ViT-B/16 train imgs/s", "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
            "ms_per_step": ms / steps, "scaling": "weak", "dtype": "bf16", "global_batch": batch * world,
            "parallelism": f"dp{world}: batch {batch}/GPU, NCCL gradient all-reduce per block bucket, CUDA-graph step",
            "loss": loss_val, "gpu_launches": n_launch, "collectives": exposed,
            "algorithmic_tflops_per_gpu": tflops, "frac_of_sustained_bf16_peak": tflops / peak}


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import hba
    from hba import ops
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # stdout carries exactly one JSON line: NCCL's version banner (NCCL_DEBUG=VERSION/WARN) goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)             # (the banner is a plain printf at communicator creation)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    hba.set_precision(args.precision)
    if args.sweep_only:
        print(json.dumps(measure_sweep(args, device, world)))
        return
    model, opt = build_gpu_model(args, device)
    eng = model.clip_model.hba_engine()
    eng.cache_text = False  # the reference recomputes the text tower every step (NEW:298)
    crit = torch.nn.MSELoss()
    B = args.batch
    g = torch.Generator().manual_seed(rank)
    host_images = torch.randn(B, 3, 224, 224, generator=g).pin_memory()
    host_targets = (torch.randn(B, N_CLASSES, generator=g) * 9.5 + 5.75).pin_memory()
    dev_images, dev_targets = host_images.to(device), host_targets.to(device)

    # functions._pipeline_core.TrainStep is the step `train_model` itself runs for every batch
    # (NEW:985-1003: zero_grad, CLIPHBA forward, MSE, NaN guard, backward, AdamW): no trunk-cache ids are
    # passed, so it is the full-trunk step, replayed as a CUDA graph after its first two calls
    import functions._pipeline_core as core
    train_step = core.TrainStep.of(model, opt, crit, device)

    def step_resident():
        train_step(dev_images, dev_targets)
        return train_step.last_loss

    # e2e: every step copies ITS inputs from pinned host memory and reads its loss back, all inside the
    # timed region.  The copies run on a side stream into one of two device buffers, issued before the
    # previous step's loss is read back, so the copy of step i+1 overlaps the compute of step i (what a
    # prefetching loader does; the reference copies synchronously at the top of the step, NEW:876-877).
    copy_stream = torch.cuda.Stream(device=device)
    slots = [(torch.empty_like(dev_images), torch.empty_like(dev_targets), torch.cuda.Event()) for _ in range(2)]
    e2e_state = {"next": 0, "staged": None}

    def stage_inputs():
        img, tgt, ev = slots[e2e_state["next"]]
        e2e_state["next"] ^= 1
        # (the slot's previous reader was step i-1, whose loss has already been read back: no wait needed)
        with torch.cuda.stream(copy_stream):
            img.copy_(host_images, non_blocking=True)
            tgt.copy_(host_targets, non_blocking=True)
            ev.record(copy_stream)
        return img, tgt, ev

    def step_e2e():
        img, tgt, ev = e2e_state["staged"] or stage_inputs()
        torch.cuda.current_stream(device).wait_event(ev)
        train_step(img, tgt)
        e2e_state["staged"] = stage_inputs()          # next step's host -> device copy, overlapping this step
        return float(train_step.last_loss)            # device -> host read of the step's result

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, profile_gemm=False):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if profile_gemm:
            ops.GEMM_PROFILE = []
        c0 = ops.COUNTERS["launches"]
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        prof, ops.GEMM_PROFILE = ops.GEMM_PROFILE, None
        launches = ops.COUNTERS["launches"] - c0
        if dist is not None:
            t = torch.tensor([ms], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, launches, prof

    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local)
    sampler.start()
    ms, launches, _ = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, train_step.last_loss, model)
    # roofline of the dominant kernel: CUDA events around every GEMM launch, which needs the launches to
    # come from the host - the same K steps once more with graph replay switched off (identical kernels)
    # (and with the text tower on the main stream: overlapped kernels would stretch each other's events)
    os.environ["HBA_STEP_GRAPH"] = "0"
    os.environ["HBA_TEXT_STREAM"] = "0"
    ms_probe, _, _ = timed(step_resident, 3)
    # long enough (>= --roofline-seconds) for the clocks to settle where a training run keeps them: the
    # denominator is then MEASURED_PEAKS' sustained figure; the burst fraction is reported beside it
    roof_steps = max(args.steps, int(args.roofline_seconds * 1e3 / (ms_probe / 3)) + 1)
    roof_sampler = ClockSampler(local)
    roof_sampler.start()
    ms_eager, _, prof = timed(step_resident, roof_steps, profile_gemm=True)
    roof_clocks = roof_sampler.stop()
    os.environ.pop("HBA_STEP_GRAPH")
    # the kernel's SHARE of the step: every libhba launch of a few host-launched steps bracketed by events the
    # same way (numerator and denominator then carry the same launch-latency bias)
    os.environ["HBA_STEP_GRAPH"] = "0"
    with ops.EventProfile() as ep:
        for _ in range(3):
            step_resident()
        torch.cuda.synchronize()
    os.environ.pop("HBA_STEP_GRAPH")
    os.environ.pop("HBA_TEXT_STREAM")
    per_entry = ep.totals_ms()
    all_ms = sum(per_entry.values())
    shares = {k: round(v / all_ms, 4) for k, v in sorted(per_entry.items(), key=lambda kv: -kv[1])[:6]}
    loss_val = float(step_resident())
    for _ in range(2):
        step_e2e()
    e2e_state["staged"] = None   # the timed region issues every one of its own copies
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    clocks = sampler.stop()      # sampled over the three timed regions (value, roofline pass, e2e)

    value = world * B * args.steps / (ms / 1e3)
    e2e_value = world * B * args.steps / (ms_e2e / 1e3)
    flops = sum(2.0 * M * N * K for (M, N, K, ns, a, b) in prof)
    gemm_ms = sum(a.elapsed_time(b) for (M, N, K, ns, a, b) in prof)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        pk = json.load(open(peaks_path))
        peak, peak_burst = pk["bf16_tflops_sustained"], pk["bf16_tflops"]
        peak_src = ("measured (MEASURED_PEAKS.json bf16_tflops_sustained: the roofline pass runs "
                    f"{ms_eager / 1e3:.1f} s back to back)")
    else:
        peak, peak_burst = 1400.0, 1650.0
        peak_src = "fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)"
    achieved = flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    # which measured peak is the honest denominator is decided by the clocks of the pass itself: MEASURED_PEAKS'
    # "sustained" figure was taken at a median 1,327 MHz (power-limited cuBLAS loop); a pass whose SM clock stays
    # near its maximum is compared with the burst figure, however long it ran
    peak_sustained = peak
    mhz, mhz_max = roof_clocks.get("sm_mhz"), roof_clocks.get("sm_max_mhz")
    if mhz and mhz_max and mhz >= 0.9 * mhz_max:
        peak = peak_burst
        peak_src = (f"measured (MEASURED_PEAKS.json bf16_tflops, the burst figure: the {ms_eager / 1e3:.1f} s roofline "
                    f"pass kept the SM clock at a median {mhz:.0f} of {mhz_max:.0f} MHz)")
    shapes = {}
    for (M, N, K, ns, a, b) in prof:
        e = shapes.setdefault((M, N, K), [0, 0.0])
        e[0] += 1
        e[1] += a.elapsed_time(b)
    by_shape = [{"M": M, "N": N, "K": K, "launches_per_step": n / roof_steps, "us_per_launch": 1e3 * t / n,
                 "tflops": 2.0 * M * N * K * n / (t / 1e3) / 1e12}
                for (M, N, K), (n, t) in sorted(shapes.items(), key=lambda kv: -kv[1][1])][:12]
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "gemm_traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get("dram_bytes_per_launch")
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "bf16x3 (fp32 mode)", "data": "synthetic",
        "config": workload_config(args, world),
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                "how": "functions._pipeline_core.TrainStep on pinned-host inputs: per step one host->device copy of "
                       "the batch (side stream, double-buffered, overlapping the previous step) and one "
                       "device->host read of the loss; K+1 copies are issued inside the timed region",
                "h2d_bytes_per_step": host_images.numel() * 4 + host_targets.numel() * 4,
                "d2h_bytes_per_step": 4},
        "gpu_launches": launches, "loss": loss_val, "clocks": clocks,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05)", "achieved": achieved,
                     "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                     "peak_source": peak_src, "peak_burst": peak_burst, "frac_of_burst_peak": achieved / peak_burst,
                     "peak_sustained": peak_sustained, "frac_of_sustained_peak": achieved / peak_sustained,
                     "pass_seconds": ms_eager / 1e3, "pass_steps": roof_steps, "pass_clocks": roof_clocks,
                     "gemm_launches_per_step": len(prof) / roof_steps,
                     "gemm_flops_per_step": flops / roof_steps,
                     "gemm_ms_per_step": gemm_ms / roof_steps,
                     "gemm_share_of_step": per_entry.get("hba_gemm_bf16", 0.0) / all_ms,
                     "kernel_time_shares": shares, "eager_ms_per_step": ms_eager / roof_steps,
                     "how": "CUDA events around every gemm_tc_kernel launch over pass_steps host-launched, single-stream "
                            "steps of the same workload, run right after the timed region (which replays the step as a "
                            "CUDA graph with the text tower on a parallel branch); shares = event time per C-ABI entry "
                            "point / event time of all libhba launches of 3 further host-launched steps",
                     "by_shape": by_shape},
    }
    out["host_cpus"] = os.cpu_count()
    # The secondary sections must never cost the headline line: a failure is recorded and reported.
    if not args.no_fp32 and args.precision == "bf16":
        # the parity mode (three bf16 passes per GEMM, fp32 attention: 1e-3 of the fp32 reference) on the same
        # workload, through the same TrainStep - reported beside the bf16 headline
        try:
            hba.set_precision("fp32")
            train_step.start_epoch()      # restages the frozen weights as hi/lo operands (as every epoch start does)
            for _ in range(3):
                step_resident()
            n32 = max(3, min(args.steps, 10))
            ms32, _, _ = timed(step_resident, n32)
            out["fp32_mode"] = {"value": world * B * n32 / (ms32 / 1e3), "unit": UNIT, "ms_per_step": ms32 / n32,
                                "steps": n32, "loss": float(train_step.last_loss),
                                "what": "hba.set_precision('fp32'): 3 bf16 passes per GEMM over hi/lo split operands, "
                                        "exact fp32 attention / LayerNorm / residual"}
        except Exception as exc:
            out["fp32_mode"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        finally:
            hba.set_precision(args.precision)
            train_step.start_epoch()
    if not args.no_hbm_kernels and rank == 0:
        # north star item 3: the bandwidth-bound kernels against the measured HBM peak (CUDA events, L2 flushed)
        try:
            from tools import bench_kernels
            hk = bench_kernels.measure(device, reps=7, with_cpu=False)
            out["roofline_hbm"] = {"peak": hk["peak_hbm_gbs"], "unit": "GB/s", "timing": hk["timing"],
                                   "empty_launch_us": hk.get("empty_launch_us"),
                                   "kernels": [{"kernel": k, "us": 1e3 * v["ms"], "bytes": v["algorithmic_bytes"],
                                                "achieved": v["achieved_gbs"], "frac": v["frac_of_measured_peak"],
                                                "us_in_stream": 1e3 * v["ms_in_stream"] if "ms_in_stream" in v else None,
                                                "frac_in_stream": v.get("frac_of_measured_peak_in_stream")}
                                               for k, v in hk["kernels"].items()]}
        except Exception as exc:
            out["roofline_hbm"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if not args.no_sweep:
        del model, opt, train_step
        torch.cuda.empty_cache()
        try:
            sw = measure_sweep(args, device, world)
        except Exception as exc:
            sw = {"error": f"{type(exc).__name__}: {exc}"[:300], "sec_per_epoch_cached": float("nan")}
        if dist is not None:
            t = torch.tensor([sw["sec_per_epoch_cached"]], device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if "error" not in sw:
                sw["sec_per_epoch_cached"] = float(t)
                sw["sec_per_condition"] = (sw["sec_first_epoch_cache_fill"] + sw["sec_second_epoch_graph_capture"]
                                           + (EPOCHS_PER_CONDITION - 2) * float(t))
                sw["conditions_per_hour"] = world * 3600.0 / sw["sec_per_condition"]
                sw["blended_images_per_s"] = world * sw["images_per_epoch"] / float(t)
        # The number that counts: a slice of the 136-condition grid run FOR REAL through the scheduler
        # (hba.sweep.run_sweep: one pinned worker process per GPU, LPT queue, every condition trained until
        # the reference's early stopping ends it, all files written).  `steady_state_replica` keeps the
        # in-process epoch timing above as the explanation of where the time goes.
        torch.cuda.empty_cache()
        sched = measure_sweep_scheduler(args, world, rank, dist)
        if rank == 0:
            steady = sw
            sw = dict(sched)
            sw["steady_state_replica"] = steady
        out["sweep"] = sw
    if not args.no_vit:
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        try:
            out["vit_b16"] = measure_vit(args, device, world, dist)
        except Exception as exc:
            out["vit_b16"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        n = args.cpu_sample_images or args.batch
        step = cpu_step_fn(build_cpu_reference(args.backbone), n)
        step()  # warm-up (allocations, thread pool)
        t0 = time.perf_counter()
        reps = 2
        for _ in range(reps):
            step()
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": n * reps / dt, "unit": UNIT, "cores": torch.get_num_threads(),
                               "kind": "port", "sample_batch": n,
                               "sample": f"{reps} training steps of {n} images = the stated batch (same model, "
                                         "fwd+bwd+AdamW, text tower recomputed), oracle port in PyTorch fp32"}
        # BASELINE.md 3 "also report": the same oracle port run by PyTorch eager ON THIS B200 (library
        # kernels: cuBLAS / SDPA), fp32 and bf16 autocast, full batch - the bar a user of the reference
        # would get from `model.to('cuda')` alone.  A reported baseline, never part of the product path.
        try:
            out["cpu_baseline"]["torch_eager_same_gpu"] = eager_gpu_baseline(args, device)
        except Exception as exc:   # reporting only
            out["cpu_baseline"]["torch_eager_same_gpu"] = {"error": str(exc)[:200]}
    if rank == 0:
        print(json.dumps(out))
    sys.stdout.flush()
    if dist is not None:
        # (measure_vit closed its trainer: the captured graphs that held NCCL kernels of the communicator are
        # gone before the group is torn down.  The watchdog only guards the driver's run against a teardown hang.)
        done = threading.Event()

        def _watchdog():
            if not done.wait(60):
                sys.stderr.write("bench.py: destroy_process_group did not return within 60 s; leaving\n")
                sys.stderr.flush()
                os._exit(0)
        threading.Thread(target=_watchdog, daemon=True).start()
        torch.cuda.synchronize()
        dist.barrier()
        dist.destroy_process_group()
        done.set()


if __name__ == "__main__":
    main()
