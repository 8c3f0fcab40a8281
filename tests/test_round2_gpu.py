"""Round-2 GPU parity cases (VERDICT round 1, "What's weak" 1-3):
  * a7  QVBertModel.forward / BertEncoder.forward (PreSelect -> 6 BERT layers -> 6 x [GCP, BERT layer]) against the oracle;
  * a9  BertEncoderLayer with the +-5e4 clamps ACTIVE (hot weights drive the intermediate activations past the clamp);
  * a11 the dot-product token head alone, at the north-star 1e-3;
  * a17 the detector at the BENCHMARKED shape (one 800x1333 image, 80-class prompt, K = 5) against intermediates and
        detections recorded from the reference's own GeneralizedVLRCNN_New.forward (tests/golden/detector_bench.pt), and
        B = 8 self-consistency (image i of the batch == the B = 1 run);
  * DETECTIONS_PER_IMG = 300 (every lvis_* eval config) and the packed (detections + count) result buffer;
  * ml_nms against the reference's kernel with exact score ties.
"""
import math
import os

import pytest
import torch

from util import FP16_TOL, ROOT, assert_close, load_sd, vq_cfg

pytestmark = pytest.mark.gpu


def _iou(a, b):
    x1, y1 = torch.max(a[:, None, 0], b[None, :, 0]), torch.max(a[:, None, 1], b[None, :, 1])
    x2, y2 = torch.min(a[:, None, 2], b[None, :, 2]), torch.min(a[:, None, 3], b[None, :, 3])
    inter = (x2 - x1 + 1).clamp(min=0) * (y2 - y1 + 1).clamp(min=0)
    aa = (a[:, 2] - a[:, 0] + 1) * (a[:, 3] - a[:, 1] + 1)
    ab = (b[:, 2] - b[:, 0] + 1) * (b[:, 3] - b[:, 1] + 1)
    return inter / (aa[:, None] + ab[None] - inter)


# ---------------------------------------------------------------------------------------------------------------------
# a7
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,ncls", [(2, 10), (1, 80)])
def test_qvbert_model_vs_oracle(dev, B, ncls):
    """Whole language backbone: embeddings, PreSelect, 12 BERT layers with GCP blocks before layers 6..11, the
    ``BertEncoder`` output dict.  18 chained fp16-operand stages -> bound 3x the per-operator tolerance."""
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.language_backbone.bert_model_new import BertEncoder
    from oracle import restate, synth
    gen = synth.Gen(500 + ncls)
    sd = synth.qvbert_sd(gen)
    ids, am, pmap = synth.prompt(ncls, 2, 256, gen)
    ids, am = ids.expand(B, -1).contiguous(), am.expand(B, -1).contiguous()
    vision, vmask = synth.vision_queries(pmap, 5, 256, 256, gen)
    vision = vision.expand(B, -1, -1).contiguous() + 0.1 * gen.randn(B, vision.shape[1], 256)
    vmask = vmask.expand(B, -1, -1).contiguous()
    I = 1117 if ncls == 10 else 5577  # the real pooled-pyramid length of an 800x1344 image on the 80-class case
    images = gen.randn(B, I, 256)
    ref = restate.qvbert_model(ids, am, vision, images, vmask, sd)
    enc = BertEncoder(mq_glip_t_cfg())
    load_sd(enc.model, sd)
    enc = enc.to(dev).eval()
    out = enc({"input_ids": ids.to(dev), "attention_mask": am.to(dev),
               "vision_inputs": {"vision": vision.to(dev), "images": images.to(dev), "vision_attention_mask": vmask.to(dev),
                                 "batched_pos_category_map": None}})
    assert set(out) >= {"aggregate", "embedded", "masks", "hidden", "vision_query_gates"}
    bad = []
    assert_close(out["hidden"], ref["hidden"], 3e-3, f"QVBertModel hidden B={B} ncls={ncls}", defer=bad)
    assert_close(out["embedded"], ref["embedded"], 3e-3, "QVBertModel embedded", defer=bad)
    assert_close(out["aggregate"], ref["aggregate"], 3e-3, "QVBertModel aggregate", defer=bad)
    assert torch.equal(out["masks"].cpu(), am)
    assert len(out["vision_query_gates"]["ffn_gates"]) == 6
    assert not bad, bad


# ---------------------------------------------------------------------------------------------------------------------
# a9
# ---------------------------------------------------------------------------------------------------------------------
def test_bert_encoder_layer_clamps_active(dev):
    """BertEncoderLayer (vldyhead.py:250-301) with weights hot enough that BertIntermediate and BertOutput exceed +-5e4:
    the clamps (rpn/modeling_bert.py:250-271) decide the result.  Also checks that BertSelfOutput is NOT clamped."""
    from types import SimpleNamespace
    from mqdet_b200.modeling.rpn.vldyhead import BertEncoderLayer
    from oracle import restate, synth
    gen = synth.Gen(43)
    sd = synth.bert_layer_sd(gen, "")
    sd["intermediate.dense.weight"] = sd["intermediate.dense.weight"] * 1.0e5      # |intermediate| ~ 1.4e5 > 5e4
    sd["output.dense.weight"] = sd["output.dense.weight"] * 1.0e-3
    B, T, D = 2, 256, 768
    h = gen.randn(B, T, D)
    am = torch.ones(B, T)
    am[0, 180:] = 0
    ref = restate.bert_layer(h, restate.extended_mask(am), sd, "", clamp=50000.0)
    unclamped = restate.bert_layer(h, restate.extended_mask(am), sd, "", clamp=0.0)
    assert (ref - unclamped).abs().max().item() > 1e-2, "the case must make the clamps matter"
    cfg = SimpleNamespace(hidden_size=D, num_attention_heads=12, intermediate_size=3072, layer_norm_eps=1e-12)
    layer = load_sd(BertEncoderLayer(cfg, clamp_min_for_underflow=True, clamp_max_for_overflow=True), sd).to(dev).eval()
    out = layer({"visual": None, "lang": {"hidden": h.to(dev), "masks": am.to(dev)}})["lang"]["hidden"]
    assert_close(out, ref, 2e-3, "BertEncoderLayer with active clamps")
    # normal magnitudes: clamps inert, the layer equals the plain BERT layer at the per-operator tolerance
    sd2 = synth.bert_layer_sd(synth.Gen(44), "")
    ref2 = restate.bert_layer(h, restate.extended_mask(am), sd2, "", clamp=50000.0)
    layer2 = load_sd(BertEncoderLayer(cfg, True, True), sd2).to(dev).eval()
    out2 = layer2({"visual": None, "lang": {"hidden": h.to(dev), "masks": am.to(dev)}})["lang"]["hidden"]
    assert_close(out2, ref2, what="BertEncoderLayer, clamps inert")


# ---------------------------------------------------------------------------------------------------------------------
# a11
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,N", [(2, 751), (1, 22400)])
def test_dot_product_head_alone(dev, B, N):
    """vldyhead.py:806-818,871-888 in isolation: normalize, 768->256 projection of e/2, token bias, region x token product,
    1/exp(log_scale), +-5e4 clamp — at the north-star tolerance (1e-3 of max|ref|)."""
    from mqdet_b200 import ops
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.rpn.vldyhead import VLDyHead
    from oracle import restate, synth
    gen = synth.Gen(610 + B)
    sd = synth.vldyhead_sd(gen, 0)
    sd["log_scale"] = torch.tensor([0.37])
    T = 256
    feat = gen.randn(B, N, 256)
    hidden = gen.randn(B, T, 768)
    masks = torch.ones(B, T, dtype=torch.long)
    ref = restate.dot_product_head(feat.half().float(), hidden, sd)   # the tower hands the head fp16 features
    head = load_sd(VLDyHead(mq_glip_t_cfg(**{"MODEL.DYHEAD.NUM_CONVS": 0})), sd).to(dev).eval()
    sizes = [(N, 1)]
    r = head.forward_flat(feat.half().to(dev).contiguous(), ops.Levels(sizes, dev), hidden.to(dev), masks.to(dev))
    assert r["dot_product_logits"].dtype == torch.float32
    assert_close(r["dot_product_logits"], ref, FP16_TOL, f"dot-product head alone N={N}")
    w = torch.cat([sd["bbox_pred.weight"].flatten(1), sd["centerness.weight"].flatten(1)])
    b = torch.cat([sd["bbox_pred.bias"], sd["centerness.bias"]])
    assert_close(r["reg_ctr"], feat.half().float() @ w.half().float().t() + b, FP16_TOL, "bbox / centerness 1x1 heads")


# ---------------------------------------------------------------------------------------------------------------------
# a17 at the benchmarked shape
# ---------------------------------------------------------------------------------------------------------------------
def _bench_model(dev, c):
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    model = GeneralizedVLRCNN_New(mq_glip_t_cfg())
    full = dict(c["sd"])
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            full[k] = v
    model = load_sd(model, full).to(dev).eval()
    model.query_selector.set_query_bank(c["bank"])
    return model


def test_detector_at_benchmark_shape_vs_reference_golden(dev):
    """ONE 800x1333 image (padded 800x1344: N = 22400 locations, I = 5577 pooled tokens), 80-class prompt (V = 400), K = 5:
    the per-image workload of BASELINE config 2, against sub-sampled intermediates and the detections of the REFERENCE's own
    forward executed on CPU (oracle/make_golden.py detector_bench).  Exercises the multi-wave / tile-edge paths of the
    B-resident GEMM at M = 22400 per image and the 88-step fused attention loop."""
    from mqdet_b200.structures.image_list import ImageList
    from oracle import make_golden
    c = make_golden.case_inputs("detector_bench")
    fx = torch.load(os.path.join(ROOT, "tests", "golden", "detector_bench.pt"))
    model = _bench_model(dev, c)
    il = ImageList(c["img"].to(dev), [c["size"]])
    caps = {"input_ids": c["ids"], "attention_mask": c["am"]}
    out = model.forward_device(il, caps, c["pmap"])
    bad = []

    def cmp(key, got, tol):
        g = make_golden.sub(got.float().cpu(), *fx["subsample"][key])
        err = (g - fx[key]).abs().max().item()
        bound = tol * fx[key + "_absmax"] + tol
        from util import _records
        _records.append(dict(what=f"bench-shape golden {key}", max_abs_err=err, bound=bound, ref_absmax=fx[key + "_absmax"],
                             rel=err / fx[key + "_absmax"]))
        if err > bound:
            bad.append(f"{key}: {err:.3e} > {bound:.3e}")

    head = out["head"]
    cmp("pyramid", out["pyramid16"], 4e-3)
    cmp("lang_hidden", out["lang_hidden"], 4e-3)
    cmp("logits", head["dot_product_logits"], 1.5e-2)
    want = fx["det"]
    res = model(il, captions=caps, positive_map=c["pmap"])[0].to("cpu")
    assert res.size == (1333, 800)
    iou = _iou(want[:, :4], res.bbox)
    same = want[:, 5, None] == res.get_field("labels")[None].float()
    matched = ((iou > 0.9) & same & ((want[:, 4, None] - res.get_field("scores")[None]).abs() < 2e-2)).any(1)
    frac = matched.float().mean().item()
    if frac < 0.85:
        bad.append(f"only {frac:.2f} of the {want.shape[0]} reference detections matched")
    assert not bad, bad


def test_batch8_equals_single_image_runs(dev):
    """BASELINE config 2 runs B = 8 images per step: image i of the batch must equal the B = 1 run of image i (no
    cross-image leakage through batched tiles, span scheduling, group statistics or the batched NMS)."""
    from mqdet_b200.structures.image_list import ImageList
    from oracle import make_golden, synth
    c = make_golden.case_inputs("detector_bench")
    model = _bench_model(dev, c)
    B = 8
    imgs = synth.images(synth.Gen(73), B, 800, 1333)
    caps = {"input_ids": c["ids"], "attention_mask": c["am"]}
    out8 = model.forward_device(ImageList(imgs.to(dev), [c["size"]] * B), caps, c["pmap"])
    lg8 = out8["head"]["dot_product_logits"].clone()
    det8, num8 = out8["det"].clone(), out8["num"].clone()
    for i in (0, 5):
        o1 = model.forward_device(ImageList(imgs[i:i + 1].to(dev), [c["size"]]), caps, c["pmap"])
        assert_close(lg8[i:i + 1], o1["head"]["dot_product_logits"], 1e-4, f"image {i}: batch-of-8 logits vs single")
        assert int(num8[i]) == int(o1["num"][0])
        k = int(num8[i])
        assert_close(det8[i, :k], o1["det"][0, :k], 1e-4, f"image {i}: detections")


# ---------------------------------------------------------------------------------------------------------------------
# DETECTIONS_PER_IMG = 300, packed result
# ---------------------------------------------------------------------------------------------------------------------
def test_detections_per_img_300_and_packed_result(dev):
    from mqdet_b200 import parallel
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.structures.image_list import ImageList
    from oracle import restate, synth
    gen = synth.Gen(2025)
    sd = synth.detector_sd(gen, bias0=-1.0)
    ids, am, pmap = synth.prompt(10, 2, 256, gen)
    bank = synth.query_bank(pmap, 5, gen)
    B, h, w = 2, 160, 224
    img = synth.images(gen, B, h, w)
    ref = restate.detector(img, (h, w), ids, am, pmap, bank, sd, max_det=300)
    model = GeneralizedVLRCNN_New(mq_glip_t_cfg(**{"MODEL.ATSS.DETECTIONS_PER_IMG": 300}))
    full = dict(sd)
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            full[k] = v
    model = load_sd(model, full).to(dev).eval()
    model.query_selector.set_query_bank(bank)
    assert model.max_out() == 352
    il = ImageList(img.to(dev), [(h, w)] * B)
    caps = {"input_ids": ids, "attention_mask": am}
    out = model.forward_device(il, caps, pmap)
    assert out["det"].shape == (B, 352, 6) and out["det_packed"].shape == (B, 353, 6)
    det_u, num_u = parallel.unpack(out["det_packed"])
    assert torch.equal(num_u.cpu(), out["num"].cpu()) and torch.equal(det_u, out["det"])
    res = model(il, captions=caps, positive_map=pmap)
    for b in range(B):
        # (1) exact: NMS + top-300 of the DEVICE candidates == the oracle's select_over_all_levels on those very candidates
        n = int(out["cand_totals"][b])
        gb, gs, gl = out["cand_boxes"][b, :n].cpu(), out["cand_scores"][b, :n].cpu(), out["cand_labels"][b, :n].cpu()
        keep_ref = restate.select_over_all_levels(gb, gs, gl, 0.6, 300)
        num = int(out["num"][b])
        assert num == keep_ref.numel() and torch.equal(out["keep"][b, :num].cpu(), keep_ref)
        assert torch.equal(out["det"][b, :num, :4].cpu(), gb[keep_ref]) and torch.equal(out["det"][b, :num, 4].cpu(), gs[keep_ref])
        assert len(res[b]) == num and torch.equal(res[b].bbox.cpu(), gb[keep_ref])
        # (2) free-running against the oracle's own forward.  The synthetic weights give every location ten near-identical
        # class scores and many overlapping boxes within 1e-3 of each other, so the ~1e-3 score noise of the fp16 tower flips
        # NMS winners (ten detections per flip, measured 3-7 flips per image: tools/dbg_match.py) and moves the top-300 cut;
        # a flipped winner still overlaps the oracle's winner by more than the NMS threshold.  Hence: same label, score
        # within 2e-2, IoU > 0.5 for >= 85 % — the strict IoU > 0.9 match is asserted on the 100-detection cases
        # (test_detector_forward, test_detector_vs_reference_golden) where those ties do not dominate.
        rb, rs, rl = ref["detections"][b]
        assert rb.shape[0] > 128, "the case must keep more than the old hard 128-row limit"
        assert abs(len(res[b]) - rb.shape[0]) <= 8, (len(res[b]), rb.shape[0])
        iou = _iou(rb, res[b].bbox.cpu())
        same = rl[:, None] == res[b].get_field("labels").cpu()[None]
        matched = ((iou > 0.5) & same & ((rs[:, None] - res[b].get_field("scores").cpu()[None]).abs() < 2e-2)).any(1)
        assert matched.float().mean().item() >= 0.85, matched.float().mean().item()
    # a too-small result buffer is an error, never a silent truncation
    from mqdet_b200._lib import MqdetError
    small = model.forward_device(il, caps, pmap, max_out=64)
    with pytest.raises(MqdetError):
        model.rpn.to_boxlists(small["det"], small["num"], [(h, w)] * B)


def test_prompt_cache_invalidation(dev):
    """ADVICE round 1: swapping the bank, editing positive_map in place or passing new token ids must not reuse stale state."""
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from oracle import synth
    gen = synth.Gen(9)
    model = GeneralizedVLRCNN_New(mq_glip_t_cfg(**{"MODEL.DYHEAD.NUM_CONVS": 1})).to(dev).eval()
    ids, am, pmap = synth.prompt(4, 2, 256, gen)
    caps = {"input_ids": ids, "attention_mask": am}
    model.query_selector.set_query_bank(synth.query_bank(pmap, 5, gen))
    s1 = model._prompt_state(caps, pmap, 1, dev)
    assert model._prompt_state(caps, pmap, 1, dev) is s1
    v1 = s1["vision"].clone()
    model.query_selector.set_query_bank(synth.query_bank(pmap, 5, gen))   # new bank, same prompt objects
    s2 = model._prompt_state(caps, pmap, 1, dev)
    assert s2 is not s1 and not torch.equal(s2["vision"], v1)
    pmap[1] = [1]                                                          # in-place edit of the positive map
    s3 = model._prompt_state(caps, pmap, 1, dev)
    assert s3 is not s2 and not torch.equal(s3["vmask"], s2["vmask"])
    ids[0, 1] += 1                                                         # in-place edit of the token ids
    s4 = model._prompt_state(caps, pmap, 1, dev)
    assert s4 is not s3 and int(s4["ids"][0, 1]) == int(ids[0, 1])


# ---------------------------------------------------------------------------------------------------------------------
# ml_nms vs the reference kernel with exact score ties
# ---------------------------------------------------------------------------------------------------------------------
def test_ml_nms_score_ties_equal_reference_kernel(dev):
    """Exact ties between boxes of DIFFERENT labels (ties inside a label would make the reference's unstable device sort
    decide the result): kept set bit-identical to csrc/cuda/ml_nms.cu."""
    from test_nms_gpu import _boxes
    from test_ref_kernels_gpu import _ref
    from mqdet_b200 import ops
    from util import reference_outputs
    n, nlabels = 3000, 40
    boxes, _, _ = _boxes(4242, n, nlabels)
    g = torch.Generator().manual_seed(5)
    scores = torch.rand(n // 2, generator=g).unique()
    m = scores.numel()
    scores = torch.cat([scores, scores])                     # every score appears exactly twice
    labels = torch.cat([torch.randint(1, nlabels // 2 + 1, (m,), generator=g),
                        torch.randint(nlabels // 2 + 1, nlabels + 1, (m,), generator=g)]).float()   # ... on different labels
    boxes = boxes[: 2 * m]
    # the reference kernel's kept set, stored under tests/golden/reference/ref_kernels.pt
    want = reference_outputs("ref_kernels", "ml_nms_score_ties",
                             lambda: {"keep": _ref().ml_nms(boxes.to(dev), scores.to(dev), labels.to(dev), 0.6)}, full=("keep",))["keep"]
    got = ops.ml_nms(boxes.to(dev), scores.to(dev), labels.to(dev), 0.6).cpu()
    assert torch.equal(got, want)


# ---------------------------------------------------------------------------------------------------------------------
# chunked many-category evaluation (LVIS path) on a small case
# ---------------------------------------------------------------------------------------------------------------------
def test_chunked_forward_equals_per_chunk_forwards_and_oracle(dev):
    """27 classes in chunks of 10 (3 prompts, the last one shorter; token positions differ per chunk): the batched-chunk path
    (backbone once, chunks as batch elements, per-element positive maps + label tables) must return, per image, the
    concatenation of what one whole forward per chunk returns (the reference's loop, engine/inference.py:605-625), and match
    the oracle run chunk by chunk."""
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.structures.image_list import ImageList
    from oracle import restate, synth
    gen = synth.Gen(2026)
    sd = synth.detector_sd(gen, bias0=-1.0)
    chunks = synth.chunked_prompts(27, 10, 256, gen)
    bank = {}
    for _, _, pm in chunks:
        bank.update(synth.query_bank(pm, 5, gen))
    B, h, w = 2, 160, 224
    img = synth.images(gen, B, h, w)
    cfg = mq_glip_t_cfg(**{"MODEL.ATSS.DETECTIONS_PER_IMG": 300})
    model = GeneralizedVLRCNN_New(cfg)
    full = dict(sd)
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            full[k] = v
    model = load_sd(model, full).to(dev).eval()
    model.query_selector.set_query_bank(bank)
    il = ImageList(img.to(dev), [(h, w)] * B)
    caps = [{"input_ids": i, "attention_mask": a} for i, a, _ in chunks]
    pmaps = [pm for _, _, pm in chunks]
    merged = model.forward_chunked(il, caps, pmaps, chunks_per_pass=2)
    assert len(merged) == B
    # (1) == one whole forward per chunk, concatenated
    for b in range(B):
        parts = []
        for cap, pm in zip(caps, pmaps):
            # per-chunk forward with the same compact column order: labels must be remapped the same way, so compare through
            # the chunked API restricted to one chunk (one pass = one chunk)
            parts.append(model.forward_chunked(il, [cap], [pm], chunks_per_pass=1)[b])
        boxes = torch.cat([p.bbox for p in parts])
        labels = torch.cat([p.get_field("labels") for p in parts])
        scores = torch.cat([p.get_field("scores") for p in parts])
        assert len(merged[b]) == boxes.shape[0]
        assert torch.equal(merged[b].get_field("labels"), labels)
        assert_close(merged[b].bbox, boxes, 1e-4, f"chunk batching, image {b}: boxes")
        assert_close(merged[b].get_field("scores"), scores, 1e-4, f"chunk batching, image {b}: scores")
    # (2) vs the oracle, chunk by chunk (labels are the GLOBAL class ids of each chunk)
    for b in range(B):
        rb, rs, rl = [], [], []
        for (ids, am, pm) in chunks:
            local = {j + 1: pm[c] for j, c in enumerate(sorted(pm))}          # oracle columns 1..n in ascending label order
            lbank = {j + 1: bank[c] for j, c in enumerate(sorted(pm))}
            ref = restate.detector(img[b:b + 1], (h, w), ids, am, local, lbank, sd, num_classes=len(local), max_det=300)
            bx, sc, lb = ref["detections"][0]
            glob = torch.tensor(sorted(pm))[lb.long() - 1]
            rb.append(bx); rs.append(sc); rl.append(glob)
        rb, rs, rl = torch.cat(rb), torch.cat(rs), torch.cat(rl)
        assert set(merged[b].get_field("labels").tolist()) <= set(range(1, 28))
        assert abs(len(merged[b]) - rb.shape[0]) <= max(8, rb.shape[0] // 20), (len(merged[b]), rb.shape[0])
        iou = _iou(rb, merged[b].bbox)
        same = rl[:, None] == merged[b].get_field("labels")[None]
        matched = ((iou > 0.9) & same & ((rs[:, None] - merged[b].get_field("scores")[None]).abs() < 2e-2)).any(1)
        assert matched.float().mean().item() >= 0.85, f"image {b}: {matched.float().mean().item():.2f} matched"


# ---------------------------------------------------------------------------------------------------------------------
# f3: vision-query extraction (extract_query: expand -> level mapping -> aligned ROIAlign 7x7 -> mean -> bank)
# ---------------------------------------------------------------------------------------------------------------------
def test_extract_query_vs_oracle(dev, tmp_path):
    """GeneralizedVLRCNN_New.extract_query on the GPU (one fused level-mapping + ROIAlign + mean kernel over the fp16 pyramid)
    against the oracle, which is pinned to the reference's own extract_query (tests/test_oracle_pinning.py); boxes on several
    FPN levels, a degenerate box removed by the clipping, MAX_QUERY_NUMBER and the bank round trip through its file format."""
    from collections import defaultdict
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.modeling.poolers import Pooler
    from mqdet_b200.structures.bounding_box import BoxList
    from mqdet_b200.structures.image_list import ImageList
    from oracle import make_golden, restate, synth
    c = make_golden.case_inputs("detector")
    model = GeneralizedVLRCNN_New(mq_glip_t_cfg())
    full = dict(c["sd"])
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            full[k] = v
    model = load_sd(model, full).to(dev).eval()
    gen = synth.Gen(556)
    W_, H_ = 896, 640
    img = synth.images(gen, 2, H_, W_)
    boxes = [torch.tensor([[10., 12., 40., 50.], [100., 60., 330., 300.], [0., 0., 895., 639.], [200., 100., 203., 104.],
                           [880., 620., 895., 639.], [895.9, 5., 896., 60.], [300., 200., 620., 500.]]),
             torch.tensor([[30., 30., 190., 200.], [5., 200., 80., 318.], [300., 20., 820., 590.]])]
    labels = [torch.tensor([3, 1, 2, 3, 7, 9, 5]), torch.tensor([1, 1, 4])]
    targets = []
    for b, l in zip(boxes, labels):
        t = BoxList(b.clone(), (W_, H_), mode="xyxy")
        t.add_field("labels", l)
        targets.append(t)
    bank = model.extract_query(images=ImageList(img.to(dev), [(H_, W_)] * 2), targets=targets, query_images=defaultdict(list))
    pyr = restate.fpn(restate.swin_transformer(img, restate._sub(c["sd"], "backbone.body.")), restate._sub(c["sd"], "backbone.fpn."))
    ex, lab = [], []
    for b, l in zip(boxes, labels):
        nb, keep = restate.expand_boxes(b.clone(), (W_, H_), 1.5)
        ex.append(nb)
        lab.append(l[keep])
    feats, lvls = restate.pool_query_features(pyr, ex)
    assert len(set(lvls.tolist())) >= 3
    lab = torch.cat(lab)
    assert sorted(bank) == sorted(set(lab.tolist()))
    for label in bank:
        want = feats[lab == label][:, None, :]
        assert bank[label].shape == want.shape and bank[label].dtype == torch.float32
        assert_close(bank[label], want, 4e-3, f"extract_query label {label}")      # the pyramid itself is 4e-3 (fp16 backbone)
    # the pooler alone on fp16-exact features: the kernel's level mapping + aligned ROIAlign at the per-operator tolerance
    pyr16 = [p.half().float() for p in pyr]
    pl = Pooler((7, 7), (0.125, 0.0625, 0.03125, 0.015625, 0.0078125), 0, use_v2=True)
    tg = model.expand_bbox(targets, 1.5)
    got = pl([p.to(dev) for p in pyr16], tg)
    from torchvision.ops import roi_align
    assert got.shape == (lab.numel(), 256, 7, 7)
    f2, l2 = restate.pool_query_features(pyr16, ex)
    assert_close(got.mean(dim=[-2, -1]), f2, 1e-3, "Pooler (level mapping + aligned ROIAlign)")
    # MAX_QUERY_NUMBER and the on-disk format (tools/extract_vision_query.py: torch.save of {label: [n, 1, C]})
    b2 = model.extract_query(images=ImageList(img.to(dev), [(H_, W_)] * 2), targets=targets, query_images=defaultdict(list),
                             max_query_number=1)
    assert all(v.shape[0] == 1 for v in b2.values())
    path = os.path.join(tmp_path, "bank.pth")
    model.save_query_bank(bank, path)
    model.load_query_bank(path)
    assert sorted(model.query_selector.query_bank) == sorted(bank)
    assert torch.equal(model.query_selector.query_bank[1].cpu(), bank[1])
