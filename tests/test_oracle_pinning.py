"""CPU: pins oracle/restate.py against the reference's own modules, through their outputs on seeded inputs stored under
tests/golden/reference/oracle_pinning.pt (recorded where the reference's sources are present: see util.reference_outputs)."""
import sys

import pytest
import torch

from oracle import make_golden, ref_loader, restate, synth
from util import ref_close, ref_equal, ref_pair, reference_outputs


def _close(a, b, tol=2e-5):
    ref_close(a, b, tol)


def _ref(case, compute, full=()):
    return reference_outputs("oracle_pinning", case, compute, full)


def test_gcp_block_vs_reference():
    c = make_golden.case_inputs("gcp_block")

    def compute():
        out = make_golden.run_reference("gcp_block")
        # the index table of the reference's topk-based construction (modeling_bert_new.py:40-63)
        out["idx"] = ref_loader.modeling_bert_new().get_index_with_padding_batch(c["mask"].transpose(2, 1))
        return out
    ref = _ref("gcp_block", compute)
    _close(restate.gcp_block(c["x"], c["vision"], c["mask"], c["sd"]), ref["y"])
    _close(restate.gcp_sparse_attention(c["x"], c["vision"], c["mask"], c["sd"], "attn."), ref["s"])
    assert ref_equal(restate.gcp_index(c["mask"]), ref["idx"])


def test_preselect_vs_reference():
    c = make_golden.case_inputs("preselect")
    _close(restate.preselect(c["vision"], c["image"], c["sd"]), _ref("preselect", lambda: make_golden.run_reference("preselect"))["vision"])


def test_bi_attention_vs_reference():
    c = make_golden.case_inputs("bi_attention")
    ref = _ref("bi_attention", lambda: make_golden.run_reference("bi_attention"))
    v = torch.cat([f.flatten(2).transpose(1, 2) for f in c["feats"]], dim=1)
    v2, l2 = restate.bi_attention(v, c["l"], c["mask"], c["sd"])
    _close(v2, ref["v"])
    _close(l2, ref["l"])


def test_bert_layer_vs_reference():
    c = make_golden.case_inputs("bert_layer")
    ref = _ref("bert_layer", lambda: make_golden.run_reference("bert_layer"))
    _close(restate.bert_layer(c["h"], restate.extended_mask(c["am"]), c["sd"], "", clamp=50000.0), ref["h"])


def test_swin_fpn_vs_reference():
    c = make_golden.case_inputs("swin_fpn")
    ref = _ref("swin_fpn", lambda: make_golden.run_reference("swin_fpn"))
    outs = restate.swin_transformer(c["img"], c["sd"])
    for i, o in enumerate(outs):
        _close(o, ref[f"c{i + 2}"], 1e-5)
    for i, o in enumerate(restate.fpn(outs, c["fsd"])):
        _close(o, ref[f"p{i + 3}"], 1e-5)


def test_swin_l_vs_reference():
    """Swin-L geometry of MQ-GLIP-L (window 12, embed 192, heads 6/12/24/48; depths shortened to 2,2,2,2 to keep the CPU
    run short): the oracle's swin_transformer with ws=12 against the reference's own SwinTransformer."""
    import torch
    from oracle import ref_loader as rl
    from oracle import synth
    gen = synth.Gen(1240)
    depths, heads, embed, ws = (2, 2, 2, 2), (6, 12, 24, 48), 192, 12
    sd = synth.swin_sd(gen, depths=depths, heads=heads, embed=embed, ws=ws)
    img = gen.randn(1, 3, 150, 203)

    def compute():
        sw = rl.swint()
        body = sw.SwinTransformer(embed_dim=embed, depths=list(depths), num_heads=list(heads), window_size=ws, drop_path_rate=0.0,
                                  frozen_stages=-1, use_checkpoint=False)
        body.eval()
        full = dict(sd)
        for k, v in body.state_dict().items():
            if k.endswith("relative_position_index"):
                full[k] = v
        body.load_state_dict(full, strict=True)
        with torch.no_grad():
            return {"outs": body(img)}
    ref = _ref("swin_l", compute)["outs"]
    with torch.no_grad():
        outs = restate.swin_transformer(img, sd, depths=depths, heads=heads, embed=embed, ws=ws)
    assert len(outs) == len(ref)
    for o, r in zip(outs, ref):
        _close(o, r, 1e-5)


def test_contrastive_embed_vs_reference():
    c = make_golden.case_inputs("contrastive_embed")
    ref = _ref("contrastive_embed", lambda: make_golden.run_reference("contrastive_embed"))["logits"]
    got = restate.contrastive_embed(c["x"], c["y"], c["mask"], 256)
    assert got.shape == (2, 900, 256)
    g, r = ref_pair(got, ref)
    assert torch.equal(torch.isinf(g), torch.isinf(r))              # padding tokens and columns T..255 are -inf
    # the same fp32 product; recorded on another CPU, whose BLAS may order the sums differently
    _close(got, ref)


def test_atss_postprocess_vs_reference():
    """ATSSPostProcessor.forward (rpn/inference.py:592-769) — sigmoid, MEAN token->class aggregation, 0.05 threshold,
    per-level top-1000, BoxCoder.decode, clip, sqrt score, ml_nms over all levels, kthvalue cut at 100 — run from the
    reference's own file on CPU, with only the compiled ml_nms kernel substituted (by the oracle's restatement of it, which
    is pinned against the real kernel on the GPU).  The oracle's post-processing must produce the same detections."""
    gen = synth.Gen(41)
    sizes, strides = [(20, 28), (10, 14), (5, 7), (3, 4), (2, 2)], [8, 16, 32, 64, 128]
    B, T, C = 2, 256, 80
    img_w, img_h = 28 * 8, 20 * 8
    _, _, pmap = synth.prompt(C, 2, T, gen)
    regs = [gen.randn(B, 4, h, w) for h, w in sizes]
    ctrs = [gen.randn(B, 1, h, w) for h, w in sizes]
    dots = [gen.randn(B, h * w, T, scale=1.5) - 2.0 for h, w in sizes]          # ~6 % of (location, class) pairs pass 0.05
    anc = [restate.anchors_level(h, w, s, 8.0 * s) for (h, w), s in zip(sizes, strides)]

    def compute():
        inf = ref_loader.rpn_inference(lambda b, s, l, t: restate.ml_nms(b, s, l, t))
        BoxList = sys.modules["maskrcnn_benchmark.structures.bounding_box"].BoxList
        coder = sys.modules["maskrcnn_benchmark.modeling.box_coder"].BoxCoder(weights=(10.0, 10.0, 5.0, 5.0))
        post = inf.ATSSPostProcessor(pre_nms_thresh=0.05, pre_nms_top_n=1000, nms_thresh=0.6, fpn_post_nms_top_n=100, min_size=0,
                                     num_classes=C + 1, box_coder=coder, score_agg="MEAN")
        cls = [torch.zeros(B, C, h, w) for h, w in sizes]
        anchors = [[BoxList(a.clone(), (img_w, img_h), mode="xyxy") for a in anc] for _ in range(B)]
        with torch.no_grad():
            ref = post(regs, ctrs, anchors, cls, None, dots, pmap)
        return {"det": [torch.cat([r.bbox, r.get_field("scores")[:, None], r.get_field("labels")[:, None].float()], 1) for r in ref]}
    ref = _ref("atss_postprocess", compute, full=("det",))["det"]
    assert any(len(r) == 100 for r in ref) or all(len(r) > 0 for r in ref)
    for b in range(B):
        parts = [restate.atss_level_candidates(dots[l][b], regs[l][b].permute(1, 2, 0).reshape(-1, 4), ctrs[l][b].reshape(-1),
                                               anc[l], pmap, C, img_w, img_h) for l in range(len(sizes))]
        assert parts[0]["boxes"].shape[0] == 1000                                   # level 0 exercises the top-k
        boxes = torch.cat([p["boxes"] for p in parts])
        scores = torch.cat([p["scores"] for p in parts])
        labels = torch.cat([p["labels"] for p in parts])
        keep = restate.select_over_all_levels(boxes, scores, labels, 0.6, 100)
        got = torch.cat([boxes[keep], scores[keep, None], labels[keep, None].float()], 1)
        want = ref[b]
        assert got.shape == want.shape, (got.shape, want.shape)

        def canon(x):  # detection order is implementation-defined (topk(sorted=False)): compare as sets
            key = x[:, 4].double() * 1e6 + x[:, 5].double() * 1e-3 + x[:, 0].double() * 1e-9
            return x[torch.argsort(key)]
        assert torch.allclose(canon(got), canon(want), rtol=1e-6, atol=1e-5)


def test_qvbert_encoder_loop_vs_reference():
    """QVBertEncoder.forward (modeling_bert_new.py:545-639) — WHICH layers get a GCP block, in which order, with which
    masks — executed from the reference's own class.  transformers 5.x changed ``BertLayer.forward``'s positional
    signature, so the twelve HF layers the encoder builds are replaced by adapters around the reference's in-repo BERT
    copy (rpn/modeling_bert.py: the same post-LN layer, itself pinned by test_bert_layer_vs_reference); the GCP blocks,
    the loop and the mask plumbing are the reference's."""
    from transformers import BertConfig
    gen = synth.Gen(51)
    sd = synth.qvbert_sd(gen)
    config = BertConfig()
    B, T = 2, 256
    _, _, pmap = synth.prompt(10, 2, T, gen)
    _, vmask = synth.vision_queries(pmap, 5, T, 768, gen)
    vmask = vmask.expand(B, -1, -1).clone()
    vmask[1, 10:20] = 0
    vq = gen.randn(B, vmask.shape[1], 768)
    h = gen.randn(B, T, 768)
    am = torch.ones(B, T)
    am[0, 180:] = 0
    ext = restate.extended_mask(am)

    def compute():
        enc = _ref_qvbert_encoder(config)
        enc.load_state_dict({k: sd["encoder." + k] for k in enc.state_dict()}, strict=True)
        with torch.no_grad():
            ref = enc(h, attention_mask=ext, vision=vq, vision_attention_mask=vmask).last_hidden_state
            ref_text_only = enc(h, attention_mask=ext).last_hidden_state
        return {"ref": ref, "ref_text_only": ref_text_only, "vision_effect": (ref - ref_text_only).abs().max().item()}
    r = _ref("qvbert_encoder_loop", compute)
    ref, ref_text_only = r["ref"], r["ref_text_only"]
    got, got_text_only = h, h
    for i in range(config.num_hidden_layers):
        if i >= 6:
            got = restate.gcp_block(got, vq, vmask, sd, f"encoder.qv_layer.{i - 6}.")
        got = restate.bert_layer(got, ext, sd, f"encoder.layer.{i}.", 12)
        got_text_only = restate.bert_layer(got_text_only, ext, sd, f"encoder.layer.{i}.", 12)
    _close(got, ref)
    _close(got_text_only, ref_text_only)
    assert r["vision_effect"] > 1e-3                             # the vision queries do change the text stream
    assert (got - got_text_only).abs().max().item() > 1e-3


def test_qvbert_model_vs_reference():
    """QVBertModel.forward end to end (modeling_bert_new.py:690-848): embeddings, extended mask, PreSelect BEFORE the encoder,
    the GCP/BERT loop — the reference's own class, with the twelve transformers-5 BertLayers swapped for adapters around
    the reference's in-repo BERT layer (see test_qvbert_encoder_loop_vs_reference)."""
    from transformers import BertConfig
    config = BertConfig()
    gen = synth.Gen(52)
    sd = synth.qvbert_sd(gen)
    B, T = 2, 256
    ids, am, pmap = synth.prompt(10, 2, T, gen)
    ids, am = ids.expand(B, -1).contiguous(), am.expand(B, -1).clone()
    am[1, 25:] = 0                                    # second caption truncated: padding inside the text stream
    vis, vmask = synth.vision_queries(pmap, 5, T, 256, gen)
    vis = vis.expand(B, -1, -1).contiguous()
    vmask = vmask.expand(B, -1, -1).clone()
    vmask[1, 5:10] = 0                                # one class of image 1 without exemplars
    images = gen.randn(B, 300, 256)

    def compute():
        m = ref_loader.modeling_bert_new()
        mod = m.QVBertModel(config, dim_t=768, dim_v=256, cfg=make_golden.ref_cfg(), add_pooling_layer=False).eval()
        mod.encoder.gradient_checkpointing = False
        mod.encoder.layer = _ref_qvbert_encoder(config).layer
        mod.load_state_dict(sd, strict=True)
        if not hasattr(mod.embeddings, "position_embedding_type"):  # transformers-4 BertEmbeddings attribute (BertConfig default)
            mod.embeddings.position_embedding_type = "absolute"
        if not hasattr(mod, "get_head_mask"):  # removed from PreTrainedModel in transformers 5
            mod.get_head_mask = lambda head_mask, n, *a, **k: [None] * n
        with torch.no_grad():
            ref = mod(input_ids=ids, attention_mask=am, vision=vis, images=images, vision_attention_mask=vmask)
        return {"hidden": ref.last_hidden_state, "ffn_gates": len(ref["vision_query_gates"]["ffn_gates"])}
    ref = _ref("qvbert_model", compute)
    got = restate.qvbert_model(ids, am, vis, images, vmask, sd)
    _close(got["hidden"], ref["hidden"])
    assert ref["ffn_gates"] == 6


def _ref_qvbert_encoder(config):
    """The reference's QVBertEncoder with its twelve transformers-5 BertLayers replaced by adapters with the positional interface
    of the BertLayer the reference was written against, around the reference's in-repo BERT layer (rpn/modeling_bert.py)."""
    import torch.nn as nn
    m, rb = ref_loader.modeling_bert_new(), ref_loader.rpn_modeling_bert()
    enc = m.QVBertEncoder(config, dim=768, cfg=make_golden.ref_cfg()).eval()
    enc.gradient_checkpointing = False  # attribute of the transformers-4 BertEncoder base class the reference targets

    class Layer(nn.Module):
        def __init__(self):
            super().__init__()
            self.attention = rb.BertAttention(config, False, False)
            self.intermediate = rb.BertIntermediate(config)
            self.output = rb.BertOutput(config)

        def forward(self, h, attention_mask=None, head_mask=None, enc_h=None, enc_mask=None, past=None, output_attentions=False):
            a = self.attention(h, attention_mask, None, output_attentions=False, past_key_value=None)[0]
            return (self.output(self.intermediate(a), a),)

    enc.layer = nn.ModuleList([Layer() for _ in range(config.num_hidden_layers)]).eval()
    return enc


def test_dyconv_vs_reference():
    """DyConv.forward (vldyhead.py:205-247) from the reference's own class: offset conv, mask sigmoid, which level feeds
    which deformable conv with which (re-interpreted) offsets, upsampling, GroupNorm, scale attention, DyReLU."""
    c = make_golden.case_inputs("dyconv")
    ref = _ref("dyconv", lambda: make_golden.run_reference("dyconv"))["v"]
    _close(restate.flatten_levels(restate.dyconv(c["feats"], c["sd"])), ref, 1e-4)


def test_vldyhead_vs_reference():
    """The whole VL deep-fusion head from the reference's own VLDyHead.forward (vldyhead.py:769-900): 6 x [VLFuse (MHA-B
    BiAttention) -> BertEncoderLayer -> DyConv], dot-product token head with its clamp, bbox (+ Scale) and centerness heads.
    Substituted (oracle/ref_loader.py::vldyhead): the compiled DCNv2 kernel (oracle restatement, pinned on the GPU),
    BertConfig.from_pretrained (no hub offline) and the transformers-4 `get_extended_attention_mask` helper."""
    c = make_golden.case_inputs("vldyhead")
    ref = _ref("vldyhead", lambda: {k: v for k, v in make_golden.run_reference("vldyhead").items() if k in ("per_level", "hidden")})
    ref_dots, ref_bbox, ref_ctr = ref["per_level"]
    got = restate.vl_dyhead(c["feats"], c["hidden"], c["masks"], c["sd"])
    off = 0
    for l, (h, w) in enumerate(make_golden.LEVELS_SMALL):
        _close(got["dot_product_logits"][:, off:off + h * w], ref_dots[l], 2e-4)
        _close(got["bbox_reg"][l], ref_bbox[l], 2e-4)
        _close(got["centerness"][l], ref_ctr[l], 2e-4)
        off += h * w
    _close(got["hidden"], ref["hidden"], 2e-4)


def test_anchors_vs_reference():
    """make_anchor_generator_complex + AnchorGenerator.forward (anchor_generator.py:72-181) with the mq-glip-t RPN block
    (sizes 64..1024, strides 8..128, one aspect ratio, one scale per octave): anchors and the visibility field of every
    level, from the reference's own module, against the oracle's closed form and the visibility rule of mqdet_anchors."""
    import types
    H, W = 160, 213                                             # true image size (the batch tensor is padded to 160 x 224)
    sizes = make_golden.LEVELS_SMALL

    def compute():
        ag = ref_loader.anchor_generator()
        cfg = types.SimpleNamespace(MODEL=types.SimpleNamespace(RPN=types.SimpleNamespace(
            ANCHOR_SIZES=(64, 128, 256, 512, 1024), ASPECT_RATIOS=(1.0,), ANCHOR_STRIDE=(8, 16, 32, 64, 128), STRADDLE_THRESH=0,
            OCTAVE=2.0, SCALES_PER_OCTAVE=1, USE_FPN=True)))
        gen = ag.make_anchor_generator_complex(cfg)
        il = sys.modules["maskrcnn_benchmark.structures.image_list"].ImageList(torch.zeros(1, 3, 160, 224), [(H, W)])
        ref = gen(il, [torch.zeros(1, 256, h, w) for h, w in sizes])[0]
        return {"bbox": [bl.bbox for bl in ref], "size": [list(bl.size) for bl in ref],
                "visibility": [bl.get_field("visibility").bool() for bl in ref]}
    ref = _ref("anchors", compute)
    assert len(ref["bbox"]) == len(sizes)
    for (h, w), stride, size, bbox, bsize, bvis in zip(sizes, (8, 16, 32, 64, 128), (64, 128, 256, 512, 1024), ref["bbox"],
                                                       ref["size"], ref["visibility"]):
        got = restate.anchors_level(h, w, stride, float(size))
        assert ref_equal(got, bbox)
        assert tuple(bsize) == (W, H)
        vis = (got[:, 0] >= 0) & (got[:, 1] >= 0) & (got[:, 2] < W) & (got[:, 3] < H)    # straddle_thresh = 0 (:96-110)
        assert ref_equal(vis, bvis)


def test_detector_vs_reference():
    """SURVEY.md §8 a17 (and a2): one whole eval forward of the reference's own ``GeneralizedVLRCNN_New.forward``
    (generalized_vl_rcnn_new.py:307-519) on CPU — Swin-T + FPN, label / location maps, QuerySelector,
    flatten_fpn_features, BertEncoder -> QVBertModel (PreSelect + GCP), VLDyHeadModule (tower, dot-product head, anchors,
    ATSS post-processing) -> BoxList — against ``restate.detector``.  Substitutions as documented in
    oracle/ref_loader.py::detector (two compiled kernels, transformers-4 shims, tokenizer)."""
    c = make_golden.case_inputs("detector")
    want = _ref("detector", lambda: {"det": make_golden.run_reference("detector")["det"]}, full=("det",))["det"]
    got = restate.detector(c["img"], c["size"], c["ids"], c["am"], c["pmap"], c["bank"], c["sd"], K=5, num_classes=80)
    boxes, scores, labels = got["detections"][0]
    have = make_golden.canonical_detections(torch.cat([boxes, scores[:, None], labels[:, None].float()], 1))
    assert have.shape == want.shape and want.shape[0] > 10, (have.shape, want.shape)
    assert torch.equal(want[:, 5], have[:, 5])                                       # same labels
    assert torch.allclose(want[:, 4], have[:, 4], rtol=2e-4, atol=2e-5)              # scores
    assert torch.allclose(want[:, :4], have[:, :4], rtol=0, atol=5e-2)               # boxes (pixels; image is 224 x 160)


def test_extract_query_vs_reference():
    """Vision-query extraction: the oracle's expand_boxes + pool_query_features against the reference's own
    GeneralizedVLRCNN_New.extract_query (expand_bbox -> Pooler(LevelMapper + ROIAlignV2) -> mean -> bank append) run on the
    reference's Swin-T + FPN; boxes spread over all five FPN levels, one degenerate box that the clipping removes."""
    import types
    from collections import defaultdict
    import torch
    from oracle import ref_loader as rl
    from oracle import synth
    c = make_golden.case_inputs("detector")
    gen = synth.Gen(555)
    W_, H_ = 1536, 1024
    img = synth.images(gen, 2, H_, W_)
    boxes = [torch.tensor([[10., 12., 40., 50.], [100., 60., 330., 300.], [0., 0., 1535., 1023.], [200., 100., 203., 104.],
                           [1500., 1000., 1535., 1023.], [1535.9, 5., 1536., 60.], [300., 200., 700., 600.]]),
             torch.tensor([[30., 30., 190., 200.], [5., 200., 80., 318.], [300., 20., 1220., 690.]])]
    labels = [torch.tensor([3, 1, 2, 3, 7, 9, 5]), torch.tensor([1, 1, 4])]

    def compute():
        cfg = make_golden.ref_detector_cfg()
        cfg.VISION_QUERY.EXPAND_RATIO, cfg.VISION_QUERY.MAX_QUERY_NUMBER, cfg.VISION_QUERY.SIMILARITY_THRESHOLD = 1.5, 5000, 0.85
        cfg.VISION_QUERY.SELECT_FPN_LEVEL = True
        det = rl.detector(cfg, make_golden.dcn_stub, lambda b, s, l, t: restate.ml_nms(b, s, l, t), (c["ids"], c["am"]))
        full = dict(c["sd"])
        for k, v in det.state_dict().items():
            if k not in full:
                full[k] = v
        det.load_state_dict(full, strict=True)
        pl = rl.poolers()
        det.pooler = pl.Pooler(output_size=(7, 7), scales=(0.125, 0.0625, 0.03125, 0.015625, 0.0078125), sampling_ratio=0, use_v2=True)
        BoxList = sys.modules["maskrcnn_benchmark.structures.bounding_box"].BoxList
        ImageList = sys.modules["maskrcnn_benchmark.structures.image_list"].ImageList
        targets = []
        for b, l in zip(boxes, labels):
            t = BoxList(b.clone(), (W_, H_), mode="xyxy")
            t.add_field("labels", l)
            targets.append(t)
        with torch.no_grad():
            bank = det.extract_query(images=ImageList(img, [(H_, W_)] * 2), targets=targets, query_images=defaultdict(list))
        return {"bank": {int(k): v for k, v in bank.items()}}
    bank = _ref("extract_query", compute)["bank"]
    with torch.no_grad():
        pyr = restate.fpn(restate.swin_transformer(img, restate._sub(c["sd"], "backbone.body.")), restate._sub(c["sd"], "backbone.fpn."))
    ex, lab = [], []
    for b, l in zip(boxes, labels):
        nb, keep = restate.expand_boxes(b.clone(), (W_, H_), 1.5)
        ex.append(nb)
        lab.append(l[keep])
    feats, lvls = restate.pool_query_features(pyr, ex)
    assert len(set(lvls.tolist())) >= 4, lvls            # the case spreads the boxes over the pyramid
    lab = torch.cat(lab)
    for label in sorted(set(lab.tolist())):
        got = feats[lab == label][:, None, :]
        _close(got, bank[label], 1e-5)
    assert sorted(bank) == sorted(set(lab.tolist()))


@pytest.mark.parametrize("ref_dim", [2, 4])
def test_ms_deform_attn_vs_reference(ref_dim):
    """GroundingDINO MultiScaleDeformableAttention (ms_deform_attn.py:136-352, CPU path = multi_scale_deformable_attn_pytorch):
    the oracle restatement against the reference's own module, 2-d reference points and 4-d reference boxes, padding mask."""
    import torch
    from oracle import ref_loader as rl
    from oracle import synth
    gen = synth.Gen(1300 + ref_dim)
    sd = synth.msda_sd(gen)
    shapes = [(20, 28), (10, 14), (5, 7), (3, 4)]
    B, Q, E = 2, 37, 256
    nv = sum(h * w for h, w in shapes)
    query, value = gen.randn(B, Q, E), gen.randn(B, nv, E)
    ref_pts = torch.rand(B, Q, 4, ref_dim, generator=gen.g)
    if ref_dim == 4:
        ref_pts[..., 2:] = ref_pts[..., 2:] * 0.3 + 0.05
    mask = torch.zeros(B, nv, dtype=torch.bool)
    mask[1, -40:] = True

    def compute():
        mod = rl.gdino_ms_deform_attn().MultiScaleDeformableAttention(embed_dim=E, num_heads=8, num_levels=4, num_points=4,
                                                                      batch_first=True)
        mod.load_state_dict(sd, strict=True)
        mod.eval()
        ss = torch.tensor(shapes)
        lsi = torch.cat([ss.new_zeros(1), (ss[:, 0] * ss[:, 1]).cumsum(0)[:-1]])
        with torch.no_grad():
            return {"out": mod(query, value=value, key_padding_mask=mask, reference_points=ref_pts, spatial_shapes=ss,
                               level_start_index=lsi)}
    want = _ref(f"ms_deform_attn_{ref_dim}", compute)["out"]
    with torch.no_grad():
        got = restate.ms_deform_attn(query, value, ref_pts, shapes, sd, key_padding_mask=mask)
    _close(got, want, 1e-5)


@pytest.mark.parametrize("case", ["plain", "masks", "wide"])
def test_gdino_bi_attention_vs_reference(case):
    """GroundingDINO BiAttentionBlock (fuse_modules.py:99-297; v_dim = l_dim = 256, embed 1024, 4 heads): the oracle restatement
    against the reference's own module — stable_softmax_2d (global maximum subtracted before the clamps), boolean -inf masks
    on both sides, and ("wide") scores spread over more than 5e4 so that the shifted lower clamp is ACTIVE."""
    import torch
    from oracle import ref_loader as rl
    from oracle import synth
    gen = synth.Gen(1400)
    sd = synth.bi_attention_sd(gen, v_dim=256, l_dim=256, embed=1024)
    B, N, T = 2, 203, 24
    v, l = gen.randn(B, N, 256), gen.randn(B, T, 256)
    mask_v = mask_l = None
    if case != "plain":
        mask_v = torch.zeros(B, N, dtype=torch.bool)
        mask_v[1, -31:] = True
        mask_l = torch.zeros(B, T, dtype=torch.bool)
        mask_l[0, -5:] = True
    if case == "wide":
        sd = dict(sd)
        sd["attn.v_proj.weight"] = sd["attn.v_proj.weight"] * 400.0
        sd["attn.l_proj.weight"] = sd["attn.l_proj.weight"] * 400.0

    def compute():
        mod = rl.gdino_fuse_modules().BiAttentionBlock(v_dim=256, l_dim=256, embed_dim=1024, num_heads=4, dropout=0.1, drop_path=0.1)
        mod.load_state_dict(sd, strict=True)
        mod.eval()
        with torch.no_grad():
            return dict(zip(("v", "l"), mod(v, l, attention_mask_v=mask_v, attention_mask_l=mask_l)))
    want = _ref(f"gdino_bi_attention_{case}", compute)
    want_v, want_l = want["v"], want["l"]
    with torch.no_grad():
        got_v, got_l = restate.gdino_bi_attention(v, l, sd, mask_v=mask_v, mask_l=mask_l)
    if case == "wide":  # the case must really exercise the shifted clamp
        vn = torch.nn.functional.layer_norm(v, (256,), sd["layer_norm_v.weight"], sd["layer_norm_v.bias"])
        ln = torch.nn.functional.layer_norm(l, (256,), sd["layer_norm_l.weight"], sd["layer_norm_l.bias"])
        q = (vn @ sd["attn.v_proj.weight"].t() + sd["attn.v_proj.bias"]) / 16.0
        k = ln @ sd["attn.l_proj.weight"].t() + sd["attn.l_proj.bias"]
        A = torch.einsum("bnhd,bthd->bhnt", q.view(B, N, 4, 256), k.view(B, T, 4, 256))
        assert (A - A.max()).min().item() < -50000.0
    _close(got_v, want_v, 1e-5)
    _close(got_l, want_l, 1e-5)
