"""GPU test of adapter placements beyond the reference drivers' 2 vision + 1 text (apply_dora_to_ViT is general,
NEW:484-513): hba.engine runs every block from the first adapted one on all rows, backward through MLP,
out_proj, softmax attention (hba_attention_bwd), in_proj and ln_1 of each - against the oracle model with torch
autograd.  The same cases run on the CPU restatement of libhba in tests/test_host_on_ref_lib_cpu.py (sequencing); here
the kernels are the real ones.  (File name: sorts after every other GPU test.)"""
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(600)]
DEV = torch.device("cuda:0")


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


# (native 224-pixel images only: T = 257 / 77 are the shapes every kernel involved has been run at on the B200; the
# fp32 form of more than two live vision blocks needs T <= 200 and is covered on the CPU restatement)
@pytest.mark.parametrize("blocks,adapters,res,precision,tol_loss,tol_grad", [
    ((3, 2), (3, 2), 224, "bf16", 3e-2, 1.5e-1),    # every block live, T = 257 like ViT-L/14 (all-bf16 attention backward)
    ((4, 3), (3, 2), 224, "bf16", 3e-2, 1.5e-1),    # a frozen block below the live ones in both towers
    ((4, 3), (2, 3), 224, "fp32", 1e-3, 2e-3),      # three live text blocks in the parity mode (causal fp32 attention backward)
    ((3, 2), (2, 2), 224, "bf16", 3e-2, 1.5e-1),    # two live text blocks, the last 2 vision blocks live
])
def test_general_adapter_placement_matches_the_oracle_model_on_the_device(blocks, adapters, res, precision, tol_loss,
                                                                          tol_grad):
    import hba
    from hba.optim import FusedAdamW
    from oracle import clip_ref, dora_ref
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
        product.to(DEV)
        crit = torch.nn.MSELoss()
        lo = crit(oracle(images), targets)
        lo.backward()
        opt = FusedAdamW(product.parameters(), lr=3e-4)
        lp = crit(product(images.to(DEV)), targets.to(DEV))
        lp.backward()
        torch.cuda.synchronize()
        assert abs(float(lp.detach()) - float(lo.detach())) <= tol_loss * abs(float(lo.detach()))
        named_p = [(n, p) for n, p in product.named_parameters() if p.requires_grad]
        named_o = [(n, p) for n, p in oracle.named_parameters() if p.requires_grad]
        assert [n for n, _ in named_p] == [n for n, _ in named_o] and len(named_p) == 3 * sum(adapters)
        for (n, a), (_, b) in zip(named_p, named_o):
            assert a.grad is not None and torch.isfinite(a.grad).all(), n
            err = float((a.grad.cpu() - b.grad).abs().max() / b.grad.abs().max())
            assert err <= tol_grad, (n, err)
        opt.step()                                    # 3 * (n_v + n_t) tensors through the fused AdamW
        with torch.no_grad():
            again = product(images.to(DEV))
        assert torch.isfinite(again).all()
    finally:
        hba.set_precision("bf16")
