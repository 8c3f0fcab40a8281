"""CPU: mqdet_b200.engine.prompts (category names -> caption strings + positive maps, the caller's side of the path) against the
reference's own functions (maskrcnn_benchmark/engine/inference.py:104-289, their source compiled as is — the module itself pulls in the
dataset / evaluation stack) on a REAL WordPiece tokenizer built offline from a synthetic vocabulary, and end to end into the token ids
the detector consumes."""
import ast
import os
import re
import types
from collections import defaultdict

import pytest
import torch

from oracle import ref_loader
from util import reference_outputs

WORDS = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]", ".", "person", "traffic", "light", "fire", "hydrant", "bicycle", "##s", "cat", "dog",
         "tv", "hot", "wine", "glass", "##es", "teddy", "bear", "hair", "drier", "cell", "phone", "potted", "plant", "stop", "sign", "a", "of",
         "photo", "sports", "ball", "(", ")", "_"]
NAMES = {1: "person", 2: "bicycle", 3: "traffic light", 4: "fire hydrant", 5: "stop_sign", 6: "cat", 7: "hot dog", 8: "wine glass",
         9: "teddy bear", 10: "hair drier", 11: "cell phone", 12: "potted plant", 13: "sports ball(round)", 14: "tv", 15: "bicycles"}


@pytest.fixture(scope="module")
def tokenizer(tmp_path_factory):
    from transformers import BertTokenizerFast
    d = tmp_path_factory.mktemp("tok") / "bert-base-uncased"
    d.mkdir()
    (d / "vocab.txt").write_text("\n".join(WORDS) + "\n")
    tok = BertTokenizerFast.from_pretrained(str(d))
    tok.save_pretrained(str(d))
    return tok, str(d)


def _cfg(tok_dir, chunk=-1):
    NS = types.SimpleNamespace
    return NS(DATASETS=NS(SEPARATION_TOKENS=". ", CAPTION_PROMPT=None, USE_CAPTION_PROMPT=False, USE_SUPRESS_QUERY=False, SUPRESS_QUERY=None),
              MODEL=NS(LANGUAGE_BACKBONE=NS(TOKENIZER_TYPE=tok_dir, MAX_QUERY_LEN=256), DYHEAD=NS(FUSE_CONFIG=NS(MLM_LOSS=False))),
              TEST=NS(CHUNKED_EVALUATION=chunk))


def _reference_functions():
    path = os.path.join(ref_loader.REF, "maskrcnn_benchmark", "engine", "inference.py")
    tree = ast.parse(open(path).read())
    want = {"clean_name", "create_positive_dict", "chunks", "create_queries_and_maps", "create_queries_and_maps_from_dataset",
            "create_positive_map_label_to_token_from_positive_map"}
    body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in want]
    assert {n.name for n in body} == want
    ns = {"re": re, "os": os, "torch": torch, "defaultdict": defaultdict}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    return ns


class _Dataset:
    def categories(self):
        return dict(NAMES)


@pytest.mark.parametrize("chunk", [-1, 4])
def test_prompts_vs_reference(tokenizer, chunk):
    """The reference's outputs are stored under tests/golden/reference/prompts.pt (see util.reference_outputs)."""
    from mqdet_b200.engine import prompts
    tok, tok_dir = tokenizer
    cfg = _cfg(tok_dir, chunk)
    pm = torch.zeros(3, 16)
    pm[0, 1:3] = 0.5
    pm[2, 7] = 1.0

    def compute():
        ref = _reference_functions()
        rq, rm = ref["create_queries_and_maps_from_dataset"](_Dataset(), cfg, disable_print=True)
        return {"queries": rq, "maps": [dict(x) for x in rm], "clean_name": ref["clean_name"]("sports ball(round)"),
                "label_to_token": dict(ref["create_positive_map_label_to_token_from_positive_map"](pm, plus=1))}
    ref = reference_outputs("prompts", f"chunk_{chunk}", compute)
    q, m = prompts.create_queries_and_maps_from_dataset(_Dataset(), cfg, tokenizer=tok)
    assert q == ref["queries"] and len(q) == (1 if chunk == -1 else 4)
    assert [dict(x) for x in m] == ref["maps"]
    assert "stop sign" in q[0] + "".join(q[1:]) and "sports ball" in "".join(q) and "(round)" not in "".join(q)   # clean_name
    assert prompts.clean_name("sports ball(round)") == ref["clean_name"]
    assert prompts.create_positive_map_label_to_token_from_positive_map(pm, plus=1) == ref["label_to_token"]


def test_prompts_into_token_ids(tokenizer):
    """Names -> captions -> token ids + positive maps: every label's positions hold exactly its word pieces."""
    from mqdet_b200.engine import prompts
    tok, tok_dir = tokenizer
    q, m = prompts.create_queries_and_maps_from_dataset(_Dataset(), _cfg(tok_dir, 5), tokenizer=tok)
    caps = prompts.tokenize_prompts(q, tok, max_query_len=64)
    assert len(caps) == 3 and all(c["input_ids"].shape == (1, 64) for c in caps)
    ids = caps[0]["input_ids"][0]
    assert tok.convert_ids_to_tokens(ids[m[0][3]].tolist()) == ["traffic", "light"]
    assert tok.convert_ids_to_tokens(caps[2]["input_ids"][0][m[2][15]].tolist()) == ["bicycle", "##s"]
    assert int(caps[0]["attention_mask"].sum()) == int((ids != 0).sum())


def test_detector_tokenizes_caption_strings_like_prompts(tokenizer):
    """String captions + an attached tokenizer (the reference's call form, generalized_vl_rcnn_new.py:378-383) give the detector the same
    token ids as the pre-tokenised dicts of ``tokenize_prompts``; the GroundingDINO model lower-cases and appends the final '.'."""
    from mqdet_b200.config import mq_glip_t_cfg, mq_groundingdino_t_cfg
    from mqdet_b200.engine import prompts
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.modeling.groundingdino.groundingdino import GroundingDINO
    tok, tok_dir = tokenizer
    q, _ = prompts.create_queries_and_maps_from_dataset(_Dataset(), _cfg(tok_dir, -1), tokenizer=tok)
    caps = prompts.tokenize_prompts(q, tok, max_query_len=256)
    det = GeneralizedVLRCNN_New.__new__(GeneralizedVLRCNN_New)   # only the tokenisation helper is exercised: no 277 M-parameter build
    det.cfg, det.tokenizer = mq_glip_t_cfg(), tok
    ids, am = det._tokenize(q, "cpu")
    assert torch.equal(ids, caps[0]["input_ids"]) and torch.equal(am, caps[0]["attention_mask"])
    gd = GroundingDINO.__new__(GroundingDINO)
    gd.cfg, gd.tokenizer = mq_groundingdino_t_cfg(), tok
    ids2, am2 = gd._tokenize(["Person. Traffic light"])
    ref = tok(["person. traffic light."], padding="max_length", return_tensors="pt")
    assert torch.equal(ids2, ref["input_ids"]) and torch.equal(am2, ref["attention_mask"])
