"""CPU: pins the training-side oracle pieces against the reference's own code, through its outputs on seeded inputs stored under
tests/golden/reference/train.pt (recorded where the reference's sources are present: see util.reference_outputs), and checks
the host-side parameter-group rules of mqdet_b200.solver.build against solver/build.py."""
import types

import torch

from oracle import ref_loader, restate
from util import ref_close, reference_outputs


def test_token_focal_loss_vs_reference():
    import sys
    g = torch.Generator().manual_seed(4)
    logits = torch.randn(2, 300, 256, generator=g) * 3 - 2
    targets = (torch.rand(2, 300, 256, generator=g) > 0.95).float()
    tm = torch.ones(2, 256)
    tm[0, 200:] = 0
    tm[1, 120:] = 0

    def compute():
        ref_loader._install_shims()
        sys.modules["maskrcnn_benchmark"]._C = types.SimpleNamespace()   # the CUDA-only sigmoid focal loss op is not on this path
        m = ref_loader._load_file("ref_sigmoid_focal_loss", "maskrcnn_benchmark/layers/sigmoid_focal_loss.py")
        mod = m.TokenSigmoidFocalLoss(0.25, 2.0)
        return {"loss": [mod(logits, targets, text_masks=mask, version="binary").item() for mask in (tm, None)]}
    ref = reference_outputs("train", "token_focal_loss", compute)["loss"]
    for mask, want in zip((tm, None), ref):
        got = restate.token_focal_loss(logits, targets, 0.25, 2.0, mask)
        assert abs(want - got.item()) <= 1e-6 * abs(want)


def test_gcp_block_autograd_oracle_vs_reference():
    """The backward oracle = autograd over restate.gcp_block: its gradients equal autograd over the reference's own block."""
    from oracle import make_golden, synth
    gen = synth.Gen(6)
    sd = synth.gcp_block_sd(gen)
    B, T = 2, 64
    _, _, pmap = synth.prompt(6, 2, T, gen)
    _, mk = synth.vision_queries(pmap, 5, T, 768, gen)
    mask = mk.expand(B, -1, -1).clone()
    mask[0, 3] = 0
    vision, x, dy = gen.randn(B, mask.shape[1], 768), gen.randn(B, T, 768), gen.randn(B, T, 768)

    def compute():
        blk = ref_loader.modeling_bert_new().GatedCrossAttentionBlock(dim=768, cfg=make_golden.ref_cfg())
        blk.load_state_dict(sd, strict=True)
        xr, vr = x.clone().requires_grad_(True), vision.clone().requires_grad_(True)
        blk(xr, vr, mask).backward(dy)
        return {"x": xr.grad, "vision": vr.grad, "params": {k: q.grad for k, q in blk.named_parameters()}}
    ref = reference_outputs("train", "gcp_block_autograd", compute)
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x2, v2 = x.clone().requires_grad_(True), vision.clone().requires_grad_(True)
    restate.gcp_block(x2, v2, mask, p, "").backward(dy)

    ref_close(x2.grad, ref["x"], 2e-5, "x")
    ref_close(v2.grad, ref["vision"], 2e-5, "vision")
    assert sorted(ref["params"]) == sorted(k for k in p if p[k].grad is not None)
    for k, q in ref["params"].items():
        ref_close(p[k].grad.view(q["sampled"] if isinstance(q, dict) else q.shape), q, 2e-5, k)


def test_param_group_rules():
    from mqdet_b200.solver.build import param_group_options
    NS = types.SimpleNamespace
    cfg = NS(SOLVER=NS(BASE_LR=1e-4, WEIGHT_DECAY=1e-4, LANG_LR=1e-5, BACKBONE_BODY_LR_FACTOR=1.0, BIAS_LR_FACTOR=2.0,
                       WEIGHT_DECAY_BIAS=0.0, WEIGHT_DECAY_NORM_FACTOR=1.0, GATE_LR=5e-3, QUERY_LR=1e-5))
    pre = "language_backbone.body.model."
    assert param_group_options(cfg, pre + "encoder.qv_layer.0.attn.to_q.weight") == (1e-5, 1e-4)
    assert param_group_options(cfg, pre + "encoder.qv_layer.0.ff_gate") == (1e-5, 1e-4)          # qv_layer rule wins over the gate rule
    assert param_group_options(cfg, pre + "encoder.qv_layer.0.attn.norm.bias") == (1e-5, 0.0)
    assert param_group_options(cfg, pre + "pre_select.layers.0.ff.linear1.weight") == (1e-5, 1e-4)
    assert param_group_options(cfg, "rpn.head.bias0") == (2e-4, 0.0)
