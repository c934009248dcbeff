"""CPU tests that PIN THE ORACLE: (1) against the golden fixtures produced by the reference's own code
(tests/golden, generator oracle/make_golden.py), (2) directly against the reference's classes when
/root/reference is present (authoring container only), (3) against an independent CLIP implementation
(transformers.CLIPModel with copied weights) for the un-vendored tower arithmetic."""
import os

import numpy as np
import pytest
import torch

from oracle import clip_ref, dora_ref, ops_ref, ref_loader
from oracle.synth import PROMPTS, synthetic_problem

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def gold(name):
    return torch.load(os.path.join(GOLD, name), weights_only=False)


def build_oracle_model(n_vis=2, n_txt=1, r=8, seed=123):
    sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=1)
    tokens = torch.stack([clip_ref.tokenize(p) for p in PROMPTS])
    model = dora_ref.CLIPHBARef(clip_ref.build_model(sd), tokens)
    torch.manual_seed(seed)
    dora_ref.apply_dora_ref(model, n_vis, n_txt, r=r)
    dora_ref.switch_dora_ref(model)
    return model


# ------------------------------------------------------------------ (1) oracle vs reference goldens
def test_dora_restatement_matches_reference_golden():
    g = gold("dora_layer.pt")
    lin = torch.nn.Linear(64, 48)
    with torch.no_grad():
        lin.weight.copy_(g["lin_weight"])
        lin.bias.copy_(g["lin_bias"])
    m, D = ops_ref.dora_init(lin.weight)
    assert torch.equal(m, g["m"]) and torch.equal(D, g["D"])
    A = g["A"].clone().requires_grad_(True)
    B = g["B"].clone().requires_grad_(True)
    mm = g["m"].clone().requires_grad_(True)
    W = ops_ref.dora_weight(D, A, B, mm, g["scaling"])
    assert torch.equal(W, g["W"])
    (W * g["G"]).sum().backward()
    for a, b in ((mm.grad, g["dm"]), (A.grad, g["dA"]), (B.grad, g["dB"])):
        assert torch.allclose(a, b, rtol=1e-6, atol=1e-8)
    # the module form consumes the RNG like the reference (A then B, Kaiming-uniform a=sqrt(5))
    torch.manual_seed(8)
    layer = dora_ref.DoRALayerRef(lin, r=8)
    assert torch.equal(layer.delta_D_A, g["A"]) and torch.equal(layer.delta_D_B, g["B"])
    assert torch.equal(layer.weight, g["W"])


def test_rsa_restatement_matches_reference_golden():
    g = gold("rsa_tail.pt")
    rho, p, rdm = ops_ref.rdm_and_spearman(g["emb"].numpy(), g["human_rdm"])
    assert rho == g["rho"] and p == g["p"]
    assert np.array_equal(rdm, g["model_rdm"])


def test_tiny_clip_forward_matches_reference_golden():
    g = gold("tiny_clip_forward.pt")
    prob = synthetic_problem()
    model = build_oracle_model()
    assert sum(p.numel() for p in model.parameters() if p.requires_grad) == g["n_trainable"]
    x, y = prob["train_images"][:3], prob["train_targets"][:3]
    pred = model(x)
    loss = torch.nn.functional.mse_loss(pred, y)
    loss.backward()
    assert torch.allclose(pred, g["pred"], rtol=1e-5, atol=1e-5)
    assert abs(float(loss) - g["loss"]) < 1e-5 * abs(g["loss"])
    params = dict(model.named_parameters())
    assert set(g["grads"]) == {n for n, p in params.items() if p.requires_grad}
    for n, gr in g["grads"].items():
        assert torch.equal(params[n].detach(), g["dora_init"][n]), n  # same RNG consumption order
        assert torch.allclose(params[n].grad, gr, rtol=1e-4, atol=1e-7), n


# ------------------------------------------------------------------ (2) oracle vs the reference itself
def test_reference_classes_equal_oracle_restatements():
    """The restated DoRALayer and CLIP-HBA model against what the reference's own classes produced
    (tests/golden/dora_layer.pt, tiny_clip_forward.pt; oracle/make_golden.py) and, where the reference tree is
    present, against those classes themselves."""
    g = gold("dora_layer.pt")
    lin = torch.nn.Linear(64, 48)
    with torch.no_grad():
        lin.weight.copy_(g["lin_weight"])
        lin.bias.copy_(g["lin_bias"])
    torch.manual_seed(8)
    layer = dora_ref.DoRALayerRef(lin, r=8)
    for n, k in (("m", "m"), ("D", "D"), ("delta_D_A", "A"), ("delta_D_B", "B")):
        assert torch.equal(getattr(layer, n), g[k]), n
    assert torch.equal(layer.weight, g["W"]) and layer.scaling == g["scaling"]
    t = gold("tiny_clip_forward.pt")
    ora = build_oracle_model()
    trainable = [(n, p) for n, p in ora.named_parameters() if p.requires_grad]
    assert [n for n, _ in trainable] == list(t["dora_init"])
    for n, p in trainable:
        assert torch.equal(p.detach(), t["dora_init"][n]), n
    assert t["n_trainable"] == sum(p.numel() for _, p in trainable) == 2 * (256 + 8 * 256 * 2) + (128 + 8 * 128 * 2)
    x = synthetic_problem()["train_images"][:t["n_images"]]
    assert torch.allclose(ora(x), t["pred"], rtol=1e-5, atol=1e-5)
    if not ref_loader.reference_available():
        return
    NEW, BASE = ref_loader.load_reference()
    torch.manual_seed(3)
    lin = torch.nn.Linear(96, 80)
    torch.manual_seed(4)
    a = NEW.DoRALayer(lin, r=16)
    torch.manual_seed(4)
    b = dora_ref.DoRALayerRef(lin, r=16)
    torch.manual_seed(4)
    c = BASE.DoRALayer(lin, r=16)
    for n in ("m", "D", "delta_D_A", "delta_D_B", "bias"):
        assert torch.equal(getattr(a, n), getattr(b, n)) and torch.equal(getattr(a, n), getattr(c, n)), n
    assert torch.equal(a.weight, b.weight) and a.scaling == b.scaling == 1.0
    # reference CLIPHBA + apply_dora_to_ViT + switch_dora_layers vs the oracle's
    ref_model = NEW.CLIPHBA(PROMPTS, backbone_name="ViT-tiny/14", pos_embedding=True)
    torch.manual_seed(123)
    NEW.apply_dora_to_ViT(ref_model, n_vision_layers=2, n_transformer_layers=1, r=8)
    NEW.switch_dora_layers(ref_model)
    ora = build_oracle_model()
    pr, po = dict(ref_model.named_parameters()), dict(ora.named_parameters())
    assert list(pr) == list(po)
    for n in pr:
        assert torch.equal(pr[n], po[n]) and pr[n].requires_grad == po[n].requires_grad, n
    x = synthetic_problem()["test_images"][:2]
    assert torch.equal(ref_model(x), ora(x))
    assert NEW.count_trainable_parameters(ref_model) == 2 * (256 + 8 * 256 * 2) + (128 + 8 * 128 * 2)


def test_reference_trainable_parameter_count_for_vit_l14_shapes():
    """183,040 trainable parameters (RUNLOG:57) = rank-32 DoRA on two 1024-wide and one 768-wide
    out_proj — checked on bare Linear layers to avoid building the 428 M parameter model: the restated layer (its
    tensors pinned against the reference's by tests/golden/dora_layer.pt), the product's, and the reference's own
    where the reference tree is present."""
    import hba
    classes = [dora_ref.DoRALayerRef, hba.DoRALayer]
    if ref_loader.reference_available():
        classes.append(ref_loader.load_reference()[0].DoRALayer)
    for cls in classes:
        n = 0
        for width in (1024, 1024, 768):
            layer = cls(torch.nn.Linear(width, width), r=32)
            n += layer.m.numel() + layer.delta_D_A.numel() + layer.delta_D_B.numel()
        assert n == 183040, cls


# ------------------------------------------------------------------ (3) independent cross-check
def test_clip_restatement_matches_transformers_clip():
    tr = pytest.importorskip("transformers")
    arch = clip_ref.ARCH["ViT-tiny/14"]
    sd = clip_ref.synthetic_state_dict("ViT-tiny/14", seed=5)
    ours = clip_ref.build_model(sd).float()
    cfg = tr.CLIPConfig(
        text_config=dict(vocab_size=arch["vocab_size"], hidden_size=arch["transformer_width"],
                         intermediate_size=4 * arch["transformer_width"],
                         num_hidden_layers=arch["transformer_layers"],
                         num_attention_heads=arch["transformer_heads"], max_position_embeddings=77,
                         hidden_act="quick_gelu", layer_norm_eps=1e-5, eos_token_id=49407,
                         bos_token_id=49406, pad_token_id=0, projection_dim=arch["embed_dim"]),
        vision_config=dict(hidden_size=arch["vision_width"], intermediate_size=4 * arch["vision_width"],
                           num_hidden_layers=arch["vision_layers"],
                           num_attention_heads=arch["vision_width"] // 64, image_size=224,
                           patch_size=arch["vision_patch_size"], hidden_act="quick_gelu",
                           layer_norm_eps=1e-5, projection_dim=arch["embed_dim"]),
        projection_dim=arch["embed_dim"])
    hf = tr.CLIPModel(cfg).eval()
    hsd = hf.state_dict()

    def put(name, value):
        assert hsd[name].shape == value.shape, (name, hsd[name].shape, value.shape)
        hsd[name] = value.clone()

    def tower(prefix_ours, prefix_hf, layers, width):
        for i in range(layers):
            o, h = f"{prefix_ours}.resblocks.{i}", f"{prefix_hf}.encoder.layers.{i}"
            w, b = sd[f"{o}.attn.in_proj_weight"], sd[f"{o}.attn.in_proj_bias"]
            for j, nm in enumerate(("q_proj", "k_proj", "v_proj")):
                put(f"{h}.self_attn.{nm}.weight", w[j * width:(j + 1) * width])
                put(f"{h}.self_attn.{nm}.bias", b[j * width:(j + 1) * width])
            put(f"{h}.self_attn.out_proj.weight", sd[f"{o}.attn.out_proj.weight"])
            put(f"{h}.self_attn.out_proj.bias", sd[f"{o}.attn.out_proj.bias"])
            for a, bb in (("ln_1", "layer_norm1"), ("ln_2", "layer_norm2"), ("mlp.c_fc", "mlp.fc1"),
                          ("mlp.c_proj", "mlp.fc2")):
                put(f"{h}.{bb}.weight", sd[f"{o}.{a}.weight"])
                put(f"{h}.{bb}.bias", sd[f"{o}.{a}.bias"])

    tower("visual.transformer", "vision_model", arch["vision_layers"], arch["vision_width"])
    tower("transformer", "text_model", arch["transformer_layers"], arch["transformer_width"])
    put("vision_model.embeddings.class_embedding", sd["visual.class_embedding"])
    put("vision_model.embeddings.patch_embedding.weight", sd["visual.conv1.weight"])
    put("vision_model.embeddings.position_embedding.weight", sd["visual.positional_embedding"])
    put("vision_model.pre_layrnorm.weight", sd["visual.ln_pre.weight"])
    put("vision_model.pre_layrnorm.bias", sd["visual.ln_pre.bias"])
    put("vision_model.post_layernorm.weight", sd["visual.ln_post.weight"])
    put("vision_model.post_layernorm.bias", sd["visual.ln_post.bias"])
    put("visual_projection.weight", sd["visual.proj"].t())
    put("text_model.embeddings.token_embedding.weight", sd["token_embedding.weight"])
    put("text_model.embeddings.position_embedding.weight", sd["positional_embedding"])
    put("text_model.final_layer_norm.weight", sd["ln_final.weight"])
    put("text_model.final_layer_norm.bias", sd["ln_final.bias"])
    put("text_projection.weight", sd["text_projection"].t())
    put("logit_scale", sd["logit_scale"])
    hf.load_state_dict(hsd)
    g = torch.Generator().manual_seed(0)
    img = torch.randn(2, 3, 224, 224, generator=g)
    tok = clip_ref.tokenize(PROMPTS[:4])
    with torch.no_grad():
        want = hf(input_ids=tok, pixel_values=img, attention_mask=None).logits_per_image
        got = ours(img, tok, True)
    assert torch.allclose(got, want, rtol=1e-4, atol=1e-3), float((got - want).abs().max())


def test_vit_restatement_matches_torchvision():
    """oracle/vit_ref.py (timm ViT restated) against an independent implementation of the same
    published architecture — torchvision's VisionTransformer — with copied weights: logits and
    parameter gradients agree to fp32 round-off."""
    from torchvision.models.vision_transformer import VisionTransformer as TVViT
    from oracle import vit_ref
    ours = vit_ref.create_model("vit_tiny_test", num_classes=10, seed=3)
    with torch.no_grad():   # give biases / norms non-trivial values
        for p in ours.parameters():
            if p.ndim == 1:
                p.add_(torch.randn_like(p) * 0.1)
    tv = TVViT(image_size=224, patch_size=16, num_layers=2, num_heads=2, hidden_dim=128, mlp_dim=512,
               num_classes=10)
    sd = {"conv_proj.weight": ours.patch_embed.proj.weight, "conv_proj.bias": ours.patch_embed.proj.bias,
          "class_token": ours.cls_token, "encoder.pos_embedding": ours.pos_embed,
          "encoder.ln.weight": ours.norm.weight, "encoder.ln.bias": ours.norm.bias,
          "heads.head.weight": ours.head.weight, "heads.head.bias": ours.head.bias}
    for i, blk in enumerate(ours.blocks):
        p = f"encoder.layers.encoder_layer_{i}."
        sd.update({p + "ln_1.weight": blk.norm1.weight, p + "ln_1.bias": blk.norm1.bias,
                   p + "self_attention.in_proj_weight": blk.attn.qkv.weight,
                   p + "self_attention.in_proj_bias": blk.attn.qkv.bias,
                   p + "self_attention.out_proj.weight": blk.attn.proj.weight,
                   p + "self_attention.out_proj.bias": blk.attn.proj.bias,
                   p + "ln_2.weight": blk.norm2.weight, p + "ln_2.bias": blk.norm2.bias,
                   p + "mlp.0.weight": blk.mlp.fc1.weight, p + "mlp.0.bias": blk.mlp.fc1.bias,
                   p + "mlp.3.weight": blk.mlp.fc2.weight, p + "mlp.3.bias": blk.mlp.fc2.bias})
    tv.load_state_dict({k: v.detach().clone() for k, v in sd.items()}, strict=True)
    tv.eval()
    ours.eval()
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 3, 224, 224, generator=g)
    y = torch.tensor([3, 7])
    lo = torch.nn.functional.cross_entropy(ours(x), y)
    lt = torch.nn.functional.cross_entropy(tv(x), y)
    assert abs(float(lo) - float(lt)) < 1e-5 * abs(float(lt))
    lo.backward()
    lt.backward()
    tvp = dict(tv.named_parameters())
    for k, p in sd.items():
        a, b = p.grad, tvp[k].grad
        assert float((a - b).abs().max()) <= 2e-4 * float(b.abs().max()) + 1e-8, k


def test_vit_schedule_matches_reference_class():
    """cosine_warmup_lr against the reference's own CosineAnnealingLRWithWarmup (VIT:206-244) when
    /root/reference is present, else against its closed form."""
    import math
    from oracle import vit_ref
    lrs = [vit_ref.cosine_warmup_lr(0.1, e, 5, 100) for e in range(100)]
    assert lrs[0] == pytest.approx(0.02) and lrs[4] == pytest.approx(0.1)
    assert lrs[5] == pytest.approx(0.1) and lrs[99] == pytest.approx(0.05 * (1 + math.cos(math.pi * 94 / 95)))
    from hba.vit import CosineAnnealingLRWithWarmup

    class _Opt:
        param_groups = [{"lr": 0.1}]
    opt = _Opt()
    sch = CosineAnnealingLRWithWarmup(opt, 5, 100)
    got = []
    for e in range(100):
        sch.step()
        got.append(opt.param_groups[0]["lr"])
    assert got == pytest.approx(lrs)
