"""Same-box speed comparators (BASELINE.md §3, SURVEY.md §2.3 / §8d; VERDICT round 1 "missing" item 6) — measurements recorded
as a GPU test because only tests/ may touch oracle/ and oracle/_ref:

  * the reference's own CUDA kernels, built unmodified for sm_100a (oracle/_ref/mqdet_ref_C.so, timed where it has been built):
    ``ml_nms`` and ``modulated_deform_conv_forward`` next to ``mqdet_ml_nms`` / ``mqdet_dcn_cols`` + the tcgen05 GEMM at the bench
    operating point ("beat the reference kernel compiled for sm_100a on the same box");
  * the reference ALGORITHM in eager PyTorch on the same B200 (oracle/restate.py moved to CUDA: the reference modules themselves
    cannot be imported on the GPU box) for one GCP block and one BiAttention fusion layer at the BASELINE config 2 shapes
    ("fused GCP kernel vs reference PyTorch attention"), fp32 and fp16 autocast.

Times: CUDA events, warm-up + 10 repetitions; written to gpurun_out/comparators.json (summarised in profiles/).
"""
import json
import os

import pytest
import torch

from util import ROOT

pytestmark = pytest.mark.gpu


def _time(fn, reps=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def _eager_bi_attention(v, l, mask_l, sd, heads=8, embed=2048):
    """The reference's BiMultiHeadAttention.forward + block residual (fuse_helper.py:218-303,419-426) as batched torch ops
    (bmm over B*heads like the reference, score matrix materialised) — the "reference PyTorch attention" comparator."""
    import torch.nn.functional as F
    B, N, _ = v.shape
    T = l.shape[1]
    d = embed // heads
    vn = F.layer_norm(v, (v.shape[-1],), sd["layer_norm_v.weight"], sd["layer_norm_v.bias"])
    ln = F.layer_norm(l, (l.shape[-1],), sd["layer_norm_l.weight"], sd["layer_norm_l.bias"])
    lin = lambda x, n: F.linear(x, sd[n + ".weight"], sd[n + ".bias"])  # noqa: E731
    sh = lambda t, n: t.view(B, n, heads, d).transpose(1, 2).reshape(B * heads, n, d)  # noqa: E731
    q, k = sh(lin(vn, "attn.v_proj") * d ** -0.5, N), sh(lin(ln, "attn.l_proj"), T)
    vv, vl = sh(lin(vn, "attn.values_v_proj"), N), sh(lin(ln, "attn.values_l_proj"), T)
    A = torch.bmm(q, k.transpose(1, 2)).clamp(min=-50000, max=50000)
    At = A.transpose(1, 2)
    Al = (At - At.max(dim=-1, keepdim=True)[0]).clamp(min=-50000, max=50000).softmax(dim=-1)
    m = torch.where(mask_l == 0, -9e15, 1.0).to(A.dtype)[:, None, None, :].expand(B, heads, N, T).reshape(B * heads, N, T)
    Av = (A + m).softmax(dim=-1)
    ov = torch.bmm(Av, vl).view(B, heads, N, d).transpose(1, 2).reshape(B, N, embed)
    ol = torch.bmm(Al, vv).view(B, heads, T, d).transpose(1, 2).reshape(B, T, embed)
    return vn + sd["gamma_v"] * lin(ov, "attn.out_v_proj"), ln + sd["gamma_l"] * lin(ol, "attn.out_l_proj")


def _eager_gcp_block(x, vision, idx, sd, heads=8, dim_head=64):
    """GatedCrossAttentionBlock.forward (modeling_bert_new.py:298-374) with the sparse MaskedCrossAttention as the reference
    runs it: K/V projected on the GATHERED [B*T, S, D] rows (the redundant projection), batched torch ops; the index table
    ``idx`` [B,T,S] (pad = V) is given (its construction is not timed)."""
    import torch.nn.functional as F
    B, T, D = x.shape
    V = vision.shape[1]
    S = idx.shape[2]
    ln = lambda t, n: F.layer_norm(t, (t.shape[-1],), sd[n + ".weight"], sd[n + ".bias"])  # noqa: E731
    vis_pad = torch.cat([vision, vision.new_zeros(B, 1, D)], dim=1)
    g = torch.gather(vis_pad, 1, idx.reshape(B, T * S, 1).expand(-1, -1, D)).view(B * T, S, D)
    xn = ln(x, "attn.norm").view(B * T, 1, D)
    kn = ln(g, "attn.norm_kv")
    inner = heads * dim_head
    q = F.linear(xn, sd["attn.to_q.weight"]) * dim_head ** -0.5
    kv = F.linear(kn, sd["attn.to_kv.weight"])
    qh = q.view(B * T, 1, heads, dim_head).transpose(1, 2)
    kh = kv[..., :inner].reshape(B * T, S, heads, dim_head).transpose(1, 2)
    vh = kv[..., inner:].reshape(B * T, S, heads, dim_head).transpose(1, 2)
    pad = (idx.reshape(B * T, 1, 1, S) == V)
    sim = qh @ kh.transpose(-1, -2) + pad.float() * -1e4
    attn = sim.softmax(dim=-1) * (~pad).float()
    s = F.linear((attn @ vh).transpose(1, 2).reshape(B, T, inner), sd["attn.to_out.weight"])
    gg = F.linear(F.gelu(F.linear(ln(s, "attn_gate.norm"), sd["attn_gate.linear1.weight"])), sd["attn_gate.linear2.weight"]).tanh()
    x1 = s * gg + x
    f = F.linear(F.gelu(F.linear(ln(x1, "ff.norm"), sd["ff.linear1.weight"])), sd["ff.linear2.weight"])
    return f * sd["ff_gate"].tanh() + x1


def test_speed_comparators(dev):
    from test_nms_gpu import _boxes
    from test_ref_kernels_gpu import _ref, _ref_dcn
    from mqdet_b200 import ops
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.language_backbone.modeling_bert_new import GatedCrossAttentionBlock
    from mqdet_b200.modeling.rpn.vldyhead import _conv_w16
    from mqdet_b200.utils.fuse_helper import BiAttentionBlockForCheckpoint
    from oracle import restate, synth
    from util import load_sd, vq_cfg
    out = {}
    # ---- ml_nms at the bench operating point: ~3600 candidates per image, 80 labels --------------------------------
    ref = _ref()
    boxes, scores, labels = _boxes(77, 3600, 80)
    scores = scores + torch.arange(3600) * 1e-7
    b, s, l = boxes.to(dev), scores.to(dev), labels.to(dev)
    out["ml_nms_3600x80"] = {"reference_kernel_ms": _time(lambda: ref.ml_nms(b, s, l, 0.6)) if ref else None,
                             "mqdet_ms": _time(lambda: ops.ml_nms_device(b, s, l, 0.6)),
                             "note": "reference = ATen sort + nms kernel + D2H of the mask + host scan (csrc/cuda/ml_nms.cu:79-149); "
                                     "mqdet = device argsort + bitmask + device scan, no D2H"}
    # ---- DCNv2 3x3 at the P3 level of a B = 8 batch (100 x 168, 256 -> 256 channels) --------------------------------
    gen = synth.Gen(5)
    B, C, H, W = 8, 256, 100, 168
    x = gen.randn(B, C, H, W).to(dev)
    om = gen.randn(B, 27, H, W, scale=1.0).to(dev)
    w = gen.randn(C, C, 3, 3, scale=0.03).to(dev)
    bias = gen.randn(C, scale=0.1).to(dev)
    off, msk = om[:, :18].contiguous(), om[:, 18:].sigmoid().contiguous()
    lv = ops.Levels([(H, W)], dev)
    x16 = x.flatten(2).transpose(1, 2).half().contiguous()
    om_flat = torch.zeros(B, H * W, 32, device=dev)
    om_flat[:, :, :27] = om.flatten(2).transpose(1, 2)
    wp = torch.nn.Parameter(w)
    w16_ = _conv_w16(wp)

    def ours():
        cols = ops.dcn_cols(x16, om_flat, lv, 1)
        return ops.gemm(cols, w16_, bias=bias)

    def ours_implicit():
        return ops.dcn_conv(x16, om_flat, lv, [1], [w16_], [bias])[0]

    y_i, y_c = ours_implicit().float(), ours().float()
    assert (y_i - y_c).abs().max().item() <= 2e-3 * y_c.abs().max().item()
    out["dcnv2_3x3_B8_100x168_256ch"] = {"reference_kernel_ms": _time(lambda: _ref_dcn(ref, x, off, msk, w, bias, 1)) if ref else None,
                                         "mqdet_ms": _time(ours_implicit), "mqdet_cols_gemm_ms": _time(ours),
                                         "note": "reference = fp32 im2col + per-image SGEMM (deform_conv_cuda.cu:496-575); "
                                                 "mqdet = implicit GEMM (mqdet_dcn_conv: sampling fused into the tcgen05 mainloop, "
                                                 "no column matrix); mqdet_cols_gemm = the fp16 NHWC sampling kernel + tcgen05 GEMM "
                                                 "pair it replaced"}
    # ---- eager-PyTorch reference algorithm vs the fused kernels: one BiAttention fusion layer, B = 8, N = 22400 ------
    sd = synth.bi_attention_sd(gen)
    blk = load_sd(BiAttentionBlockForCheckpoint(v_dim=256, l_dim=768, embed_dim=2048, num_heads=8, hidden_dim=3072, dropout=0.1,
                                                drop_path=0.0, init_values=1.0 / 6, cfg=mq_glip_t_cfg()), sd).to(dev).eval()
    Bf, N, T = 8, 22400, 256
    v32 = gen.randn(Bf, N, 256).to(dev)
    l32 = gen.randn(Bf, T, 768).to(dev)
    mask = torch.ones(Bf, T, dtype=torch.long, device=dev)
    sd_dev = {k: t.to(dev) for k, t in sd.items()}
    v16 = v32.half()
    def guarded(fn, **kw):
        try:
            return _time(fn, **kw)
        except Exception as e:  # noqa: BLE001 - a comparator that cannot run on this stack is recorded, not fatal
            torch.cuda.synchronize()
            return f"unavailable: {type(e).__name__}: {str(e)[:160]}"

    with torch.no_grad():
        t_ours = _time(lambda: blk.forward_flat(v16, l32, mask))
        # the batched eager formulation first agrees with the oracle (one image), then it is timed at B = 8
        chk_v, chk_l = _eager_bi_attention(v32[:1, :1000], l32[:1], mask[:1], sd_dev)
        ref_v, ref_l = restate.bi_attention(v32[:1, :1000].cpu(), l32[:1].cpu(), mask[:1].cpu(), sd)
        assert (chk_v.cpu() - ref_v).abs().max().item() < 1e-3 and (chk_l.cpu() - ref_l).abs().max().item() < 1e-3
        t_eager32 = guarded(lambda: _eager_bi_attention(v32, l32, mask, sd_dev), reps=3, warm=1)

        def eager16():
            with torch.autocast("cuda", dtype=torch.float16):
                return _eager_bi_attention(v32, l32, mask, sd_dev)
        t_eager16 = guarded(eager16, reps=3, warm=1)
    out["biattention_layer_B8_N22400_T256"] = {"eager_pytorch_fp32_ms": t_eager32, "eager_pytorch_fp16_autocast_ms": t_eager16,
                                               "mqdet_ms": t_ours,
                                               "note": "eager = the reference algorithm (fuse_helper.py:218-303,419-426) as torch ops on "
                                                       "the same GPU (cuBLAS + ATen softmax), materialising the score matrix"}
    # ---- one GCP block, B = 8, 80 classes x 5 queries --------------------------------------------------------------
    gsd = synth.gcp_block_sd(gen)
    _, _, pmap = synth.prompt(80, 2, 256, gen)
    _, gm = synth.vision_queries(pmap, 5, 256, 768, gen)
    gmask = gm.expand(8, -1, -1).contiguous().to(dev)
    vis = gen.randn(8, 400, 768).to(dev)
    xg = gen.randn(8, 256, 768).to(dev)
    gblk = load_sd(GatedCrossAttentionBlock(dim=768, cfg=vq_cfg()), gsd).to(dev).eval()
    gsd_dev = {k: t.to(dev) for k, t in gsd.items()}
    idx = restate.gcp_index(gm.expand(8, -1, -1)).to(dev)
    with torch.no_grad():
        chk = _eager_gcp_block(xg[:1], vis[:1], idx[:1], gsd_dev)
        refg = restate.gcp_block(xg[:1].cpu(), vis[:1].cpu(), gm, gsd)
        assert (chk.cpu() - refg).abs().max().item() < 2e-3
        t_g = _time(lambda: gblk(xg, vis, gmask))
        t_ge = guarded(lambda: _eager_gcp_block(xg, vis, idx, gsd_dev), reps=5, warm=2)
    out["gcp_block_B8_80cls"] = {"eager_pytorch_fp32_ms": t_ge, "mqdet_ms": t_g,
                                 "note": "eager = modeling_bert_new.py:298-374 as torch ops incl. the redundant per-token K/V "
                                         "projection of the reference's sparse path"}
    path = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(path):
        json.dump(out, open(os.path.join(path, "comparators.json"), "w"), indent=1)
    print(json.dumps(out))
    assert out["ml_nms_3600x80"]["mqdet_ms"] > 0
