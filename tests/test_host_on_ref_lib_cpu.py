"""The product's host side run on the CPU restatement of the C-ABI (oracle/libhba_ref.py): every libhba entry point is
served by a torch formula on host memory, so hba/ops.py, hba/engine.py (forward, live-sub-graph backward, frozen-trunk
cache), hba/dora.py, hba/optim.py, hba/rsa.py and the drop-in pipelines execute unmodified without a GPU.  What is
checked here is the SEQUENCING around the kernels - against the oracle model, and against the reference's own
`run_behavioral_training` executed on the CPU.  The kernels themselves are the `-m gpu` tests' subject."""
import csv
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
pytestmark = pytest.mark.timeout(900)


def _models(precision, r=8):
    import hba
    from oracle import clip_ref, dora_ref
    from src.models.CLIPs.clip_hba import clip as pclip
    hba.set_precision(precision)
    sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1)
    tokens = torch.stack([clip_ref.tokenize(p) for p in ("metallic; artificial", "food-related", "animal-related",
                                                         "textile", "plant-related")])
    oracle = dora_ref.CLIPHBARef(clip_ref.build_model(sd), tokens)
    torch.manual_seed(123)
    dora_ref.apply_dora_ref(oracle, 2, 1, r=r)
    dora_ref.switch_dora_ref(oracle)
    product = dora_ref.CLIPHBARef(pclip.build_model(sd), tokens)
    torch.manual_seed(123)
    dora_ref.apply_dora_ref(product, 2, 1, r=r, layer_cls=hba.DoRALayer)
    dora_ref.switch_dora_ref(product, layer_cls=hba.DoRALayer)
    return oracle, product


@pytest.mark.parametrize("precision,tol_loss,tol_grad", [("fp32", 2e-5, 2e-4), ("bf16", 5e-3, 5e-2)])
def test_engine_sequencing_matches_the_oracle_model(precision, tol_loss, tol_grad):
    """One training step of the tiny CLIP-HBA through hba.engine / hba.DoRALayer / FusedAdamW on the CPU restatement
    of libhba: predictions, loss, the 9 DoRA gradients and the updated parameters against the oracle model with
    torch autograd and torch.optim.AdamW; then the same batch served from the frozen-trunk cache, bit for bit."""
    import hba
    from hba.engine import TrunkCache
    from hba.optim import FusedAdamW
    from oracle.libhba_ref import emulated_device
    try:
        oracle, product = _models(precision)
        g = torch.Generator().manual_seed(0)
        images = torch.randn(3, 3, 224, 224, generator=g)
        targets = torch.randn(3, 5, generator=g) * 9.5 + 5.75
        crit = torch.nn.MSELoss()
        opt_o = torch.optim.AdamW([p for p in oracle.parameters() if p.requires_grad], lr=3e-3)
        po = oracle(images)
        lo = crit(po, targets)
        lo.backward()
        with emulated_device() as lib:
            opt_p = FusedAdamW(product.parameters(), lr=3e-3)
            eng = product.clip_model.hba_engine()

            def run(ids):
                for p in product.parameters():
                    p.grad = None
                eng.batch_ids = ids
                pred = product(images)
                loss = crit(pred, targets)
                loss.backward()
                return pred.detach().clone(), loss.detach().clone(), [p.grad.clone() for p in product.parameters() if p.requires_grad]
            pp, lp, grads = run(None)
            n_calls = len(lib.calls)
            eng.trunk_cache = TrunkCache(16)
            fill = run([4, 2, 9])                    # miss: trunk computed and stored
            assert eng.trunk_cache.present == {2, 4, 9}
            calls_fill = len(lib.calls) - n_calls
            hit = run([4, 2, 9])                     # hit: the frozen trunk is skipped
            calls_hit = len(lib.calls) - n_calls - calls_fill
            for a, b in ((fill, hit), ((pp, lp, grads), hit)):
                assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
                assert all(torch.equal(x, y) for x, y in zip(a[2], b[2]))
            assert calls_hit < calls_fill            # (block 0 and the attention half of block 1 were not launched)
            opt_p.step()
        opt_o.step()
        assert abs(float(lp) - float(lo.detach())) <= tol_loss * abs(float(lo.detach()))
        assert float((pp - po).abs().max() / po.abs().max()) <= tol_loss * 10
        named_p = [(n, p) for n, p in product.named_parameters() if p.requires_grad]
        named_o = [(n, p) for n, p in oracle.named_parameters() if p.requires_grad]
        assert [n for n, _ in named_p] == [n for n, _ in named_o] and len(named_p) == 9
        for (n, a), (_, b), ga in zip(named_p, named_o, grads):
            assert float((ga - b.grad).abs().max() / b.grad.abs().max()) <= tol_grad, n
            if precision == "fp32":                  # the AdamW update itself (first step: lr * sign-like step)
                assert float((a.detach() - b.detach()).abs().max()) <= 1e-5 + 1e-3 * 3e-3, n
        # the C-ABI entry points one step of this graph consists of
        assert {"hba_gemm_bf16", "hba_attention_fwd", "hba_attention_bwd_row0", "hba_dora_merge_fwd", "hba_dora_merge_bwd",
                "hba_layernorm_fwd", "hba_layernorm_bwd", "hba_cos_head_fwd", "hba_cos_head_bwd", "hba_adamw_multi",
                "hba_im2col_patches", "hba_assemble_tokens_ln", "hba_embed_tokens", "hba_gather_rows",
                "hba_add_rows"} <= set(lib.calls)
    finally:
        hba.set_precision("bf16")


def test_emulated_device_leaves_no_trace():
    """The stand-in is scoped: afterwards `is_cuda` is the real property, libhba is the real library and a CPU tensor
    is refused again (no CPU fallback in the product)."""
    import hba
    from hba import _lib, ops
    from oracle.libhba_ref import RefLib, emulated_device
    real = _lib.load()
    with emulated_device() as lib:
        assert isinstance(_lib.load(), RefLib) and _lib.load() is lib and torch.zeros(1).is_cuda
    assert _lib.load() is real and not torch.zeros(1).is_cuda
    with pytest.raises((AssertionError, RuntimeError)):
        ops.nonfinite_flag(torch.zeros(4), torch.zeros(1, dtype=torch.int32))
    assert hba.get_precision() in ("bf16", "fp32")


def test_run_behavioral_training_equals_the_reference_executed(tmp_path):
    """SURVEY 8a rows A / B / D / P / L / T / O / E / R / S / C at the level a sweep shards: the reference's OWN
    `run_behavioral_training` (BASE:707-823 and NEW:1066-1227, CPU branch) on the restated tiny CLIP against this
    repo's `run_behavioral_training` on the CPU restatement of libhba (fp32 mode, resident loaders, trunk cache,
    fused MSE, FusedAdamW), from the same image / csv / .mat / checkpoint files: a 3-epoch baseline, two conditions
    resumed from its epoch-2 checkpoints (random targets, label shuffle), one that perturbs epoch 1 from scratch, and
    two baselines with other adapter placements (2 + 2 in fp32 mode, 3 + 2 in bf16 mode: deeper live ranges).
    Losses within 2e-5 (fp32 re-association), RSA rho / p within 1e-6, and - exactly - epochs, perturbation flags,
    files, checkpoint keys, optimizer step counts and the torch / NumPy / DataLoader-generator states at the end
    (which also pins the RNG draws of the model construction, clip.replay_constructor_draws)."""
    gold = json.load(open(os.path.join(GOLD, "clip_pipeline_exec.json")))
    tool = os.path.join(ROOT, "oracle", "clip_pipeline_exec.py")
    have_reference = os.path.isdir("/root/reference/Training/functions")
    arms = ["product"] + (["reference"] if have_reference else [])
    procs = {a: subprocess.Popen([sys.executable, tool, "--arm", a, "--out", str(tmp_path / f"{a}.json")],
                                 stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for a in arms}
    for a, p in procs.items():
        out, _ = p.communicate(timeout=800)
        assert p.returncode == 0, f"{a} arm failed:\n{out[-3000:]}"
    got = json.load(open(tmp_path / "product.json"))

    def compare(want, loss_tol, rho_tol):
        assert list(got["runs"]) == list(want["runs"]) == ["baseline", "random_target", "label_shuffle",
                                                            "uniform_images_from_scratch", "baseline_2p2", "baseline_3p2"]
        for name, w in want["runs"].items():
            g = got["runs"][name]
            if name == "baseline_3p2":       # run in the bf16 mode (T = 257 is beyond the fp32 full attention backward)
                loss_tol, rho_tol = max(loss_tol, 1e-2), max(rho_tol, 1e-1)
            for k in ("last_epoch", "dora_keys", "optimizer_steps", "n_optimizer_tensors", "torch_rng_sha", "generator_sha",
                      "numpy_rng_sha", "random_state_keys", "files"):
                assert g[k] == w[k], (name, k, g[k], w[k])
            gr, wr = list(csv.reader(g["csv"].splitlines())), list(csv.reader(w["csv"].splitlines()))
            assert gr[0] == wr[0] and len(gr) == len(wr)
            for a, b in zip(gr[1:], wr[1:]):
                assert a[0] == b[0] and a[5:] == b[5:], (name, a, b)
                for i, tol in ((1, loss_tol), (2, loss_tol), (3, rho_tol), (4, rho_tol)):
                    assert abs(float(a[i]) - float(b[i])) <= tol * max(1.0, abs(float(b[i]))), (name, a, b)
            for k, (s, m) in w["dora"].items():
                if name == "baseline_3p2":   # (bf16 mode: the signed sum of a zero-mean matrix is no stable statistic)
                    assert abs(g["dora"][k][1] - m) <= 2e-2 * max(1.0, m)
                else:
                    assert abs(g["dora"][k][0] - s) <= 1e-3 * max(1.0, abs(s)) and abs(g["dora"][k][1] - m) <= 1e-3 * max(1.0, m)
    # the committed reference-arm output may come from another CPU model: losses 1e-4, rho over 28 pairs 2e-2
    compare(gold, 1e-4, 2e-2)
    rows = list(csv.reader(gold["runs"]["uniform_images_from_scratch"]["csv"].splitlines()))
    assert [r[7] for r in rows[1:]] == ["True", "False"] and gold["runs"]["random_target"]["optimizer_steps"] == [12.0]
    assert got["c_abi_calls"]["hba_gemm_bf16"] > 500 and got["c_abi_calls"]["hba_adamw_multi"] == 27 + 12
    assert len(gold["runs"]["baseline_2p2"]["dora_keys"]) == 12 and len(gold["runs"]["baseline_3p2"]["dora_keys"]) == 15
    assert got["c_abi_calls"]["hba_attention_bwd"] > 0
    if have_reference:
        compare(json.load(open(tmp_path / "reference.json")), 2e-5, 1e-6)
    # hba.rsa_scale over the baseline's DoRA checkpoints, restricted to the inference set: the rho of every checkpoint
    # is the one `train_model` wrote for that epoch (same embeddings through the cached forward, same RSA tail)
    base_rows = list(csv.reader(got["runs"]["baseline"]["csv"].splitlines()))[1:]
    scale = got["rsa_over_checkpoints"]
    assert [r["epoch"] for r in scale] == [1, 2, 3] and [r["checkpoint"] for r in scale] == [
        f"dora/epoch{e}_dora_params.pth" for e in (1, 2, 3)]
    for r, row in zip(scale, base_rows):
        assert abs(r["behavioral_rsa_rho"] - float(row[3])) < 1e-12 and abs(r["behavioral_rsa_p_value"] - float(row[4])) < 1e-12


def test_gpu_test_files_dry_run_on_the_cpu_restatement():
    """The GPU test files themselves - ops, model, pipeline, ViT - executed by pytest on the CPU with libhba served by
    its restatement (tests/emulate_clip_gpu_tests.py; captured graphs become call-by-call launches, the front ends'
    argument checks are restated; one kernel-summation-order comparison is left out).  Two things are pinned at once: the product's host side against every oracle /
    golden those tests hold, and the restatement against the formulas that judge the CUDA kernels on the B200."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emulate_clip_gpu_tests as emu
    tool = os.path.join(ROOT, "tests", "emulate_clip_gpu_tests.py")
    procs = {f: subprocess.Popen([sys.executable, tool, os.path.join(ROOT, "tests", f)], stdout=subprocess.PIPE,
                                 stderr=subprocess.STDOUT, text=True, env=dict(os.environ, OMP_NUM_THREADS="2"))
             for f in emu.DRY_RUN_FILES}
    counts = {}
    for f, p in procs.items():
        out, _ = p.communicate(timeout=800)
        assert p.returncode == 0, f"{f}:\n{out[-3000:]}"
        tail = [l for l in out.splitlines() if " passed" in l][-1]
        assert "failed" not in tail and "error" not in tail, tail
        counts[f] = int(tail.split(" passed")[0].split()[-1])
    # (the 10 streaming-LayerNorm cases of test_gpu_ops.py moved to test_gpu_rowwise_shapes.py, dry-run by
    # tests/test_rowwise_ref_cpu.py)
    assert counts["test_gpu_ops.py"] >= 86 and counts["test_gpu_pipeline.py"] >= 12, counts
    assert counts["test_gpu_model.py"] >= 6 and counts["test_gpu_vit.py"] >= 85, counts
    assert counts["test_gpu_zzz_general_placement.py"] == 4, counts


def _custom_state_dict(vision_layers, transformer_layers, seed=1):
    from oracle import clip_ref
    arch = dict(clip_ref.ARCH["ViT-tiny/14"], vision_layers=vision_layers, transformer_layers=transformer_layers)
    torch.manual_seed(seed)
    m = clip_ref.CLIP(**arch)
    with torch.no_grad():
        m.logit_scale.fill_(4.6052)
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.normal_(0, 0.02)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


@pytest.mark.parametrize("blocks,adapters,res,precision,tol", [
    ((3, 2), (3, 2), 224, "bf16", 5e-2),      # every block of the miniature live; T = 257 like ViT-L/14
    ((3, 2), (3, 2), 112, "fp32", 2e-4),      # resized positional table (T = 65): the fp32 form of the full backward
    ((4, 3), (3, 2), 112, "fp32", 2e-4),      # a frozen block below the live ones in both towers
    ((4, 3), (4, 3), 224, "bf16", 8e-2),
    ((4, 3), (3, 1), 112, "fp32", 2e-4),      # three live vision blocks, only the last text block live
    ((4, 3), (2, 3), 112, "fp32", 2e-4),      # three live text blocks, the last 2 vision blocks live
])
def test_general_adapter_placement_matches_the_oracle_model(blocks, adapters, res, precision, tol):
    """apply_dora_to_ViT(n_vision_layers, n_transformer_layers) is general (NEW:484-513); the reference drivers use
    2 + 1.  Any other placement makes more of each tower live in hba.engine (every block from the first adapted one on
    all rows, backward through MLP / out_proj / attention / in_proj / ln_1 of each) - here on the CPU restatement of libhba
    against the oracle model with torch autograd: loss and the gradients of every adapter tensor."""
    import hba
    from oracle import clip_ref, dora_ref
    from oracle.libhba_ref import emulated_device
    from src.models.CLIPs.clip_hba import clip as pclip
    try:
        hba.set_precision(precision)
        sd = _custom_state_dict(*blocks)
        tokens = torch.stack([clip_ref.tokenize(p) for p in ("metallic; artificial", "food-related", "animal-related",
                                                             "textile")])
        g = torch.Generator().manual_seed(0)
        images = torch.randn(3, 3, res, res, generator=g)
        targets = torch.randn(3, 4, generator=g) * 9.5 + 5.75
        oracle = dora_ref.CLIPHBARef(clip_ref.build_model(sd), tokens)
        torch.manual_seed(123)
        dora_ref.apply_dora_ref(oracle, *adapters, r=8)
        dora_ref.switch_dora_ref(oracle)
        product = dora_ref.CLIPHBARef(pclip.build_model(sd), tokens)
        torch.manual_seed(123)
        dora_ref.apply_dora_ref(product, *adapters, r=8, layer_cls=hba.DoRALayer)
        dora_ref.switch_dora_ref(product, layer_cls=hba.DoRALayer)
        crit = torch.nn.MSELoss()
        lo = crit(oracle(images), targets)
        lo.backward()
        with emulated_device() as lib:
            lp = crit(product(images), targets)
            lp.backward()
            with torch.no_grad():
                again = product(images)              # the no-grad forward (evaluation) runs the same blocks
        assert abs(float(lp.detach()) - float(lo.detach())) <= tol * abs(float(lo.detach()))
        assert abs(float(crit(again, targets)) - float(lp.detach())) <= 1e-6 * abs(float(lp.detach()))
        named_p = [(n, p) for n, p in product.named_parameters() if p.requires_grad]
        named_o = [(n, p) for n, p in oracle.named_parameters() if p.requires_grad]
        assert [n for n, _ in named_p] == [n for n, _ in named_o] and len(named_p) == 3 * sum(adapters)
        for (n, a), (_, b) in zip(named_p, named_o):
            assert a.grad is not None and float((a.grad - b.grad).abs().max() / b.grad.abs().max()) <= tol, n
        if max(adapters[0] - 2, adapters[1] - 1) > 0:
            assert "hba_attention_bwd" in lib.calls       # the full attention backward below the last block
    finally:
        hba.set_precision("bf16")


@pytest.mark.parametrize("vis_idx,txt_idx", [([0], [0]), ([0, 2], []), ([1], [0, 1]), ([], [0]), ([1], [])])
def test_adapters_placed_by_hand_match_the_oracle_model(vis_idx, txt_idx):
    """Placements apply_dora_to_ViT cannot produce (module surgery by hand: a frozen block ABOVE an adapted one, gaps,
    one tower only): the live range starts at the lowest adapter and the backward passes through frozen out_proj
    weights on its way down."""
    import hba
    from oracle import clip_ref, dora_ref
    from oracle.libhba_ref import emulated_device
    from src.models.CLIPs.clip_hba import clip as pclip
    try:
        hba.set_precision("fp32")
        sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1)
        tokens = torch.stack([clip_ref.tokenize(p) for p in ("metallic; artificial", "food-related", "animal-related")])
        g = torch.Generator().manual_seed(0)
        images = torch.randn(2, 3, 112, 112, generator=g)
        targets = torch.randn(2, 3, generator=g) * 9.5 + 5.75
        models = []
        for cls, builder in ((dora_ref.DoRALayerRef, clip_ref.build_model), (hba.DoRALayer, pclip.build_model)):
            m = dora_ref.CLIPHBARef(builder(sd), tokens)
            torch.manual_seed(5)
            for tower, idx in ((m.clip_model.visual.transformer, vis_idx), (m.clip_model.transformer, txt_idx)):
                for i in idx:
                    tower.resblocks[i].attn.out_proj = cls(tower.resblocks[i].attn.out_proj, r=4)
            dora_ref.switch_dora_ref(m, layer_cls=cls)
            models.append(m)
        oracle, product = models
        lo = torch.nn.functional.mse_loss(oracle(images), targets)
        lo.backward()
        with emulated_device():
            lp = torch.nn.functional.mse_loss(product(images), targets)
            lp.backward()
        assert abs(float(lp.detach()) - float(lo.detach())) <= 2e-5 * abs(float(lo.detach()))
        pg = [p.grad for p in product.parameters() if p.requires_grad]
        og = [p.grad for p in oracle.parameters() if p.requires_grad]
        assert len(pg) == len(og) == 3 * (len(vis_idx) + len(txt_idx))
        for a, b in zip(pg, og):
            assert float((a - b).abs().max() / b.abs().max()) <= 2e-4
    finally:
        hba.set_precision("bf16")


def test_fp32_mode_refuses_deep_vision_placement_at_257_tokens():
    """The fp32 form of the full attention backward holds T <= 200 tokens: three adapted vision blocks at the native
    224-pixel resolution (T = 257) are refused in the fp32 parity mode with a message, not with a kernel error."""
    import hba
    from oracle import clip_ref, dora_ref
    from oracle.libhba_ref import emulated_device
    from src.models.CLIPs.clip_hba import clip as pclip
    try:
        hba.set_precision("fp32")
        tokens = torch.stack([clip_ref.tokenize(p) for p in ("a", "b")])
        product = dora_ref.CLIPHBARef(pclip.build_model(_custom_state_dict(3, 2)), tokens)
        torch.manual_seed(1)
        dora_ref.apply_dora_ref(product, 3, 1, r=4, layer_cls=hba.DoRALayer)
        dora_ref.switch_dora_ref(product, layer_cls=hba.DoRALayer)
        with emulated_device(), pytest.raises(NotImplementedError, match="T <= 200"):
            product(torch.zeros(1, 3, 224, 224))
    finally:
        hba.set_precision("bf16")


def _abi_trace(sd, adapters, res, precisions):
    """(names + every scalar argument + which pointers are null) of all C-ABI calls of: staging, three training
    steps of the placement `adapters` = (n_vision, n_text) (no cache / cache fill / cache hit at the model's native
    resolution) with FusedAdamW, one evaluation batch - in each precision mode of `precisions`."""
    import ctypes as C
    import hba
    from hba._lib import SIGNATURES
    from hba.engine import TrunkCache
    from hba.optim import FusedAdamW
    from oracle import clip_ref, dora_ref, libhba_ref
    from src.models.CLIPs.clip_hba import clip as pclip
    trace = []

    class Tracing(libhba_ref.RefLib):
        def __getattribute__(self, name):
            fn = object.__getattribute__(self, name)
            if not name.startswith("hba_") or name == "hba_last_error":
                return fn

            def wrapped(*args):
                # pointers (by the declared argument types of hba._lib, never by value) are recorded as given / null
                if name == "hba_gemm_bf16":
                    p = args[0]._obj
                    sig = tuple(bool(getattr(p, f)) if t is C.c_void_p else getattr(p, f) for f, t in p._fields_)
                else:
                    types = SIGNATURES[name][1]
                    assert len(types) == len(args), name
                    sig = tuple(bool(libhba_ref._addr(a)) if t is C.c_void_p else a for a, t in zip(args, types))
                rc = fn(*args)
                trace.append((name, sig))
                return rc
            return wrapped
    real = libhba_ref.RefLib
    libhba_ref.RefLib = Tracing
    try:
        tokens = torch.stack([clip_ref.tokenize(p) for p in ("metallic; artificial", "food-related", "animal-related",
                                                             "textile")])
        g = torch.Generator().manual_seed(0)
        images = torch.randn(3, 3, res, res, generator=g)
        targets = torch.randn(3, 4, generator=g)
        for precision in precisions:
            hba.set_precision(precision)
            product = dora_ref.CLIPHBARef(pclip.build_model(sd), tokens)
            torch.manual_seed(123)
            dora_ref.apply_dora_ref(product, *adapters, r=8, layer_cls=hba.DoRALayer)
            dora_ref.switch_dora_ref(product, layer_cls=hba.DoRALayer)
            with libhba_ref.emulated_device():
                opt = FusedAdamW(product.parameters(), lr=3e-4)
                eng = product.clip_model.hba_engine()
                eng.trunk_cache = TrunkCache(16)
                for ids in (None, [1, 2, 3], [1, 2, 3]):
                    opt.zero_grad()
                    eng.batch_ids = ids
                    torch.nn.functional.mse_loss(product(images), targets).backward()
                    opt.step()
                with torch.no_grad():
                    eng.batch_ids = [3, 1]
                    product(images[:2])
    finally:
        libhba_ref.RefLib = real
        hba.set_precision("bf16")
    return trace


def _check_trace_golden(trace, golden):
    import hashlib
    digest = hashlib.sha256(repr(trace).encode()).hexdigest()
    path = os.path.join(GOLD, golden)
    counts = {}
    for name, _ in trace:
        counts[name] = counts.get(name, 0) + 1
    if os.environ.get("HBA_WRITE_TRACE_GOLDEN") == "1":
        with open(path, "w") as f:
            json.dump({"calls": len(trace), "sha256": digest, "per_entry": counts}, f, indent=1, sort_keys=True)
    gold = json.load(open(path))
    assert len(trace) == gold["calls"] and counts == gold["per_entry"], (len(trace), counts)
    assert digest == gold["sha256"]


def test_c_abi_call_trace_of_the_reference_placement_is_pinned():
    """The kernel sequence of the reference drivers' placement (2 vision + 1 text adapters, BDRV:28-30) is what every
    B200 measurement and GPU parity run of this repo exercised.  Its C-ABI call trace on the CPU restatement - entry
    points, shapes, leading dimensions, flags, which optional pointers are given - is pinned by a digest: a change of
    hba.engine / hba.dora / hba.optim that alters what is launched for this placement must be deliberate (regenerate:
    HBA_WRITE_TRACE_GOLDEN=1)."""
    from oracle import clip_ref
    _check_trace_golden(_abi_trace(clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1), (2, 1), 224, ("bf16", "fp32")),
                        "c_abi_trace_2p1.json")


@pytest.mark.parametrize("blocks,adapters,res,precision,golden", [
    (None, (3, 2), 224, "bf16", "c_abi_trace_3p2_bf16.json"),          # every block of the miniature live, trunk cache
    ((4, 3), (2, 3), 112, "fp32", "c_abi_trace_2p3_fp32_112.json"),    # three live text blocks above a frozen one
])
def test_c_abi_call_trace_of_deeper_placements_is_pinned(blocks, adapters, res, precision, golden):
    """The same pin for placements with live blocks below the last one: their forward keeps only what the backward
    reads, and their backward walks the live blocks down to the lowest trainable adapter."""
    from oracle import clip_ref
    sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1) if blocks is None else _custom_state_dict(*blocks)
    _check_trace_golden(_abi_trace(sd, adapters, res, (precision,)), golden)


@pytest.mark.parametrize("blocks,adapters,res,precision", [
    (None, (2, 1), 224, "bf16"),
    ((4, 3), (3, 2), 112, "fp32"),
])
def test_tower_forwards_use_disjoint_workspaces(blocks, adapters, res, precision):
    """The text tower's forward runs on a side stream concurrently with the vision tower's (HBA_TEXT_STREAM): a
    workspace both request would be raced on by the device.  Every Engine._buf key requested under the vision forward
    (vision_trunk / vision_head) must differ from every key requested under the text forward (text_features), in
    training steps with and without the trunk cache and in evaluation."""
    import inspect
    import hba
    from hba.engine import Engine, TrunkCache
    from oracle import clip_ref, dora_ref
    from oracle.libhba_ref import emulated_device
    from src.models.CLIPs.clip_hba import clip as pclip
    keys = {"vision": set(), "text": set()}
    real_buf = Engine._buf

    def recording_buf(self, name, shape, dtype=torch.float32, zero=False):
        for frame in inspect.stack(0):
            tower = {"vision_trunk": "vision", "vision_head": "vision", "text_features": "text"}.get(frame.function)
            if tower:
                keys[tower].add((name, tuple(shape), dtype))
                break
        return real_buf(self, name, shape, dtype, zero)

    sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1) if blocks is None else _custom_state_dict(*blocks)
    tokens = torch.stack([clip_ref.tokenize(p) for p in ("metallic; artificial", "food-related")])
    images = torch.randn(3, 3, res, res, generator=torch.Generator().manual_seed(0))
    try:
        hba.set_precision(precision)
        Engine._buf = recording_buf
        product = dora_ref.CLIPHBARef(pclip.build_model(sd), tokens)
        torch.manual_seed(123)
        dora_ref.apply_dora_ref(product, *adapters, r=4, layer_cls=hba.DoRALayer)
        dora_ref.switch_dora_ref(product, layer_cls=hba.DoRALayer)
        with emulated_device():
            eng = product.clip_model.hba_engine()
            eng.trunk_cache = TrunkCache(8)
            for ids in (None, [1, 2, 3], [1, 2, 3]):
                eng.batch_ids = ids
                product(images).square().mean().backward()
            with torch.no_grad():
                eng.batch_ids = [1, 2, 3]
                product(images)
    finally:
        Engine._buf = real_buf
        hba.set_precision("bf16")
    assert keys["vision"] and keys["text"]
    assert not keys["vision"] & keys["text"], sorted(keys["vision"] & keys["text"])
    assert all(k[0].startswith(("v", "keep.v")) for k in keys["vision"]), sorted(keys["vision"])
    assert all(k[0].startswith(("t", "keep.t")) for k in keys["text"]), sorted(keys["text"])
