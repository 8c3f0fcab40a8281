"""CPU, build container only: pins the GroundingDINO part of oracle/restate.py (BASELINE config 4, SURVEY.md §8 f1) against the
reference's own code — the whole ``Transformer.forward`` (encoder with fusion + text enhancer +
deformable layers, two-stage selection, decoder with iterative box refinement), ``PositionEmbeddingSineHW``, the per-category text
masks of bertwarper.py, the GroundingDINO Swin-T backbone, the BERT loop under a per-query mask with restarted position ids, and
``convert_groundingdino_to_glip_output``.  Also checks the product's host-side helpers (no GPU needed) against the same code.
The reference's outputs on the seeded inputs are stored under tests/golden/reference/gdino_pinning.pt (recorded where its
sources are present: see util.reference_outputs)."""
import ast
import os
import types
import warnings

import torch

from oracle import make_golden, ref_loader, restate, synth
from util import ref_close, ref_equal, reference_outputs

TKW = dict(d_model=256, nhead=8, dim_feedforward=2048, dropout=0.0, activation="relu", return_intermediate_dec=True, query_dim=4,
           num_feature_levels=4, enc_n_points=4, dec_n_points=4, learnable_tgt_init=True, two_stage_type="standard",
           embed_init_tgt=True, use_text_enhancer=True, use_fusion_layer=True, use_checkpoint=False, use_transformer_ckpt=False,
           use_text_cross_attention=True, text_dropout=0.0, fusion_dropout=0.0, fusion_droppath=0.1)


def _close(a, b, tol=2e-5):
    ref_close(a, b, tol)


def _ref(case, compute, full=()):
    return reference_outputs("gdino_pinning", case, compute, full)


def small_case(gen, B=2, Tt=32, used=25, shapes=((12, 16), (6, 8), (3, 4), (2, 2))):
    """Synthetic transformer inputs: 4 levels, image 1 padded on the right / bottom, a prompt of 4-token categories."""
    srcs = [gen.randn(B, 256, h, w) for h, w in shapes]
    masks = []
    for h, w in shapes:
        m = torch.zeros(B, h, w, dtype=torch.bool)
        m[1, :, int(w * 0.75):] = True
        m[1, int(h * 0.8):, :] = True
        masks.append(m)
    enc_text = gen.randn(B, Tt, 256)
    tmask = torch.ones(B, Tt, dtype=torch.bool)
    tmask[:, used:] = False
    pid = torch.zeros(B, Tt, dtype=torch.long)
    sam = torch.eye(Tt, dtype=torch.bool)[None].repeat(B, 1, 1)
    st = 1
    while st < used:
        e = min(st + 4, used)
        sam[:, st:e, st:e] = True
        pid[:, st:e] = torch.arange(e - st)
        st = e
    return srcs, masks, enc_text, tmask, pid, sam


def ref_transformer(sd, nq, enc_layers, dec_layers):
    """The reference's Transformer with its heads attached the way GroundingDINO.__init__ does (groundingdino.py:247-275)."""
    p = ref_loader.gdino_package()
    T = p.transformer.Transformer(num_queries=nq, num_encoder_layers=enc_layers, num_decoder_layers=dec_layers, **TKW).eval()
    be = p.utils.MLP(256, 256, 4, 3)
    T.decoder.bbox_embed = torch.nn.ModuleList([be for _ in range(dec_layers)])
    T.decoder.class_embed = torch.nn.ModuleList([p.utils.ContrastiveEmbed() for _ in range(dec_layers)])
    T.enc_out_bbox_embed = p.utils.MLP(256, 256, 4, 3)
    T.enc_out_class_embed = p.utils.ContrastiveEmbed()
    own = T.state_dict()
    missing = [k for k in own if k not in sd]
    assert not missing, missing[:5]
    T.load_state_dict({k: sd[k] for k in own}, strict=True)
    return T


def test_gdino_transformer_vs_reference():
    gen = synth.Gen(71)
    nq, el, dl = 20, 2, 2
    sd = synth.gdino_transformer_sd(gen, el, dl, nq=nq)
    srcs, masks, enc_text, tmask, pid, sam = small_case(gen)
    poss = [restate.position_embedding_sine_hw(m) for m in masks]

    def compute():
        T = ref_transformer(sd, nq, el, dl)
        td = {"encoded_text": enc_text.clone(), "text_token_mask": tmask, "position_ids": pid, "text_self_attention_masks": sam}
        with torch.no_grad(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            hs, refs, hs_enc, ref_enc, init = T(srcs, masks, None, poss, None, None, td)
        return {"hs": hs, "refs": refs, "text": td["encoded_text"], "padding_effect": (hs[-1][0] - hs[-1][1]).abs().max().item(),
                "fusion_effect": (td["encoded_text"] - enc_text).abs().max().item()}
    ref = _ref("transformer", compute)
    hs, refs = ref["hs"], ref["refs"]
    out = restate.gdino_transformer(srcs, masks, poss, enc_text, tmask, pid, sam, sd, num_queries=nq, enc_layers=el, dec_layers=dl)
    assert len(hs) == dl and len(refs) == dl + 1
    for a, b in zip(hs, out["hs"]):
        _close(b, a)
    for a, b in zip(refs, out["references"]):
        _close(b, a)
    _close(out["memory_text"], ref["text"])
    # the padded image differs from the un-padded one, the text stream is changed by the fusion layers
    assert ref["padding_effect"] > 1e-2 and ref["fusion_effect"] > 1e-2
    assert (out["hs"][-1][0] - out["hs"][-1][1]).abs().max() > 1e-2 and (out["memory_text"] - enc_text).abs().max() > 1e-2


def test_position_embedding_vs_reference():
    import importlib
    m = torch.zeros(2, 13, 17, dtype=torch.bool)
    m[1, 9:, :] = True
    m[1, :, 12:] = True

    def compute():
        ref_loader.gdino_package()
        pe = importlib.import_module("ref_gdino_pkg.backbone.position_encoding")
        mod = pe.PositionEmbeddingSineHW(128, temperatureH=20, temperatureW=20, normalize=True)
        misc = importlib.import_module("groundingdino_new.util.misc")
        return {"pos": mod(misc.NestedTensor(torch.zeros(2, 256, 13, 17), m))}
    ref = _ref("position_embedding", compute)["pos"]
    got = restate.position_embedding_sine_hw(m)
    assert ref_equal(got, ref)
    from mqdet_b200.modeling.groundingdino.groundingdino import PositionEmbeddingSineHW
    assert ref_equal(PositionEmbeddingSineHW(128, 20, 20)(m), ref)


def test_text_masks_vs_reference():
    import importlib
    gen = synth.Gen(72)
    ids, am, pmap = synth.prompt(13, 2, 64, gen)
    ids_b, _, _ = synth.prompt(7, 3, 64, gen)
    ids2 = torch.cat([ids, ids_b], 0)  # second row: other category lengths (the reference carries previous_col across rows)
    special = [101, 102, 1012, 1029]

    def compute():
        ref_loader.gdino_package()
        bw = importlib.import_module("ref_gdino_pkg.bertwarper")
        return dict(zip(("mask", "pos", "cate"), bw.generate_masks_with_special_tokens_and_transfer_map({"input_ids": ids2}, special, None)))
    ref = _ref("text_masks", compute, full=("mask", "pos", "cate"))
    rm, rp, rc = ref["mask"], ref["pos"], ref["cate"]
    gm, gp = restate.gdino_text_masks(ids2, special)
    assert torch.equal(gm, rm) and torch.equal(gp, rp)
    from mqdet_b200.modeling.groundingdino.bertwarper import generate_masks_with_special_tokens_and_transfer_map as mine
    pm, pp, pc = mine({"input_ids": ids2}, special)
    assert torch.equal(pm, rm) and torch.equal(pp, rp)
    assert len(pc) == len(rc) and all(torch.equal(a, b) for a, b in zip(pc, rc))
    # every category of the synthetic prompt is a block: its tokens see each other and the trailing '.', nothing else
    toks = pmap[1]
    assert rm[0, toks[0], toks[-1]] and not rm[0, toks[0], pmap[2][0]]


def test_gdino_swin_vs_reference():
    import importlib
    gen = synth.Gen(73)
    sd = synth.swin_sd(gen)
    img = synth.rgb_images(gen, 2, 75, 110)

    def compute():
        ref_loader.gdino_package()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            st = importlib.import_module("ref_gdino_pkg.backbone.swin_transformer")
            model = st.build_swin_transformer("swin_T_224_1k", 224, out_indices=(1, 2, 3), dilation=False, use_checkpoint=False)
            model.eval()  # the reference overrides train() without returning self
        own = model.state_dict()
        load = {k: sd[k] for k in own if k in sd}
        missing = [k for k in own if k not in sd and not k.endswith(("relative_position_index", "attn_mask"))]
        assert not missing, missing[:5]
        model.load_state_dict(load, strict=False)
        with torch.no_grad():
            return {"outs": model.forward_raw(img)}
    ref = _ref("swin", compute)["outs"]
    got = restate.swin_transformer(img, sd)[1:]
    assert len(ref) == 3
    for a, b in zip(ref, got):
        _close(b, a, 1e-5)


def test_bert_loop_with_category_masks_vs_reference():
    """QVBertEmbeddings with restarted position ids + the encoder loop under the [B,1,T,T] extended mask that
    get_extended_attention_mask builds from a 3-D mask (bertwarper.py:141-143), on the reference's own classes."""
    import torch.nn as nn
    from transformers import BertConfig
    config = BertConfig(num_hidden_layers=2)
    gen = synth.Gen(74)
    sd = synth.qvbert_sd(gen, layers=2, start_qv=1)
    ids, am, pmap = synth.prompt(10, 2, 64, gen)
    self_mask, pid = restate.gdino_text_masks(ids)
    ext = (1.0 - self_mask[:, None].float()) * -10000.0

    def compute():
        m, rb = ref_loader.modeling_bert_new(), ref_loader.rpn_modeling_bert()
        emb = m.QVBertEmbeddings(config, make_golden.ref_cfg()).eval()
        emb.load_state_dict({k: sd["embeddings." + k] for k in emb.state_dict() if "embeddings." + k in sd}, strict=False)
        if not hasattr(emb, "position_embedding_type"):  # transformers-4 BertEmbeddings attribute (BertConfig default)
            emb.position_embedding_type = "absolute"
        with torch.no_grad():
            ref_e = emb(input_ids=ids, position_ids=pid, token_type_ids=torch.zeros_like(ids))

        class Layer(nn.Module):
            def __init__(self):
                super().__init__()
                self.attention = rb.BertAttention(config, False, False)
                self.intermediate = rb.BertIntermediate(config)
                self.output = rb.BertOutput(config)

            def forward(self, h, attention_mask=None, head_mask=None, enc_h=None, enc_mask=None, past=None, output_attentions=False):
                a = self.attention(h, attention_mask, None, output_attentions=False, past_key_value=None)[0]
                return (self.output(self.intermediate(a), a),)

        enc = m.QVBertEncoder(config, dim=768, cfg=make_golden.ref_cfg(), start_qv_layer_index=1).eval()
        enc.gradient_checkpointing = False
        enc.layer = nn.ModuleList([Layer() for _ in range(2)]).eval()
        enc.load_state_dict({k: sd["encoder." + k] for k in enc.state_dict()}, strict=True)
        with torch.no_grad():
            return {"embeddings": ref_e, "hidden": enc(ref_e, attention_mask=ext).last_hidden_state}
    r = _ref("bert_loop_with_category_masks", compute)
    emb = restate.bert_embeddings(ids, sd, position_ids=pid)
    _close(emb, r["embeddings"])
    ref, got = r["hidden"], emb
    for i in range(2):
        got = restate.bert_layer(got, ext, sd, f"encoder.layer.{i}.", 12)
    _close(got, ref)
    full = restate.bert_layer(emb, None, sd, "encoder.layer.0.", 12)
    assert (full - restate.bert_layer(emb, ext, sd, "encoder.layer.0.", 12)).abs().max() > 1e-3  # the block mask matters


def _ref_convert_fn():
    """The reference's own ``GroundingDINO.convert_groundingdino_to_glip_output`` (groundingdino.py:291-335): the module cannot be
    imported here (tokenizer download, yacs, _C), so the method's source is compiled as is from the reference file and bound to the
    reference's own ``convert_grounding_to_od_logits`` / ``BoxList`` / ``remove_small_boxes``."""
    path = os.path.join(ref_loader.REF, "groundingdino_new", "models", "GroundingDINO", "groundingdino.py")
    tree = ast.parse(open(path).read())
    fn = None
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "convert_groundingdino_to_glip_output":
            fn = node
    assert fn is not None
    mod = ast.Module(body=[fn], type_ignores=[])
    inf = ref_loader.rpn_inference(lambda *a, **k: None)
    import sys
    ns = {"torch": torch, "convert_grounding_to_od_logits": inf.convert_grounding_to_od_logits,
          "BoxList": sys.modules["maskrcnn_benchmark.structures.bounding_box"].BoxList,
          "remove_small_boxes": sys.modules["maskrcnn_benchmark.structures.boxlist_ops"].remove_small_boxes}
    exec(compile(mod, path, "exec"), ns)
    return ns["convert_groundingdino_to_glip_output"]


def test_gdino_detections_vs_reference():
    gen = synth.Gen(75)
    B, nq, T, C = 2, 60, 256, 80
    _, am, pmap = synth.prompt(13, 2, T, gen)
    logits = gen.randn(B, nq, T, scale=2.0) - 2.0
    logits[:, :, am[0] == 0] = float("-inf")
    boxes = torch.rand(B, nq, 4, generator=gen.g)
    boxes[0, 3] = torch.tensor([0.99, 0.5, 0.3, 0.2])   # sticks out on the right: clipped
    boxes[1, 5] = torch.tensor([0.1, 0.98, 0.05, 0.3])  # sticks out at the bottom
    sizes = [(480, 640), (400, 600)]
    me = types.SimpleNamespace(cfg=types.SimpleNamespace(MODEL=types.SimpleNamespace(DYHEAD=types.SimpleNamespace(NUM_CLASSES=C + 1))),
                               box_threshold=0.05)

    def compute():
        ref = _ref_convert_fn()(me, {"pred_logits": logits.sigmoid(), "pred_boxes": boxes}, pmap, sizes)
        return {"labels": [r.get_field("labels") for r in ref], "scores": [r.get_field("scores") for r in ref], "bbox": [r.bbox for r in ref]}
    ref = _ref("detections", compute, full=("labels", "scores", "bbox"))
    got = restate.gdino_detections(logits, boxes, pmap, C, sizes, 0.05)
    assert len(got) == len(ref["labels"])
    for rl_, rs, rb, (gb, gs, gl) in zip(ref["labels"], ref["scores"], ref["bbox"], got):
        assert len(rl_) == gb.shape[0] and len(rl_) > 5
        assert torch.equal(rl_, gl)
        _close(gs, rs, 1e-6)
        _close(gb, rb, 1e-6)
