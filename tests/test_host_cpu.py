"""CPU: the host-side pieces of the drop-in boundary (no kernels) pinned against the reference's OWN classes: QuerySelector
(SURVEY.md §8 a1), BoxList, to_image_list, through their outputs on seeded inputs stored under
tests/golden/reference/host.pt (recorded where the reference's sources are present: see util.reference_outputs); plus level
tables / sharding helpers that have no reference counterpart."""
import random
import types

import numpy as np
import pytest
import torch

from oracle import ref_loader, synth
from util import ref_equal, reference_outputs


def _vq_cfg(**over):
    vq = dict(QUERY_BANK_PATH="", LEARNABLE_BANK=False, ADD_VISION_LAYER=False, PURE_TEXT_RATE=0.0, NUM_QUERY_PER_CLASS=5,
              RANDOM_KSHOT=False)
    vq.update(over)
    return types.SimpleNamespace(MODEL=types.SimpleNamespace(DEVICE="cpu"), VISION_QUERY=types.SimpleNamespace(**vq))


@pytest.mark.parametrize("training,kshot,text_rate", [(False, False, 0.0), (True, True, 0.3), (True, False, 0.0)])
def test_query_selector_vs_reference(training, kshot, text_rate):
    from mqdet_b200.modeling.query_selector.query_selector import QuerySelector
    gen = synth.Gen(7)
    _, _, pmap = synth.prompt(12, 2, 256, gen)                     # {class -> token positions}
    bank = synth.query_bank(pmap, 7, gen)                         # 7 exemplars / class, NUM_QUERY_PER_CLASS = 5 picks 5
    bank[3] = bank[3][:2]                                         # a class with fewer exemplars than requested
    labels = [sorted(bank.keys()), sorted(bank.keys())[::2]]
    T = 256
    loc = []
    for ls in labels:
        m = torch.zeros(len(ls), T)
        for i, c in enumerate(ls):
            m[i, torch.as_tensor(pmap[c])] = 1.0 / len(pmap[c])   # soft location map: the selector binarises it
        loc.append(m)
    cfg = _vq_cfg(RANDOM_KSHOT=kshot, PURE_TEXT_RATE=text_rate)

    def select(cls):
        sel = cls(cfg)
        sel.query_bank = {k: v.clone() for k, v in bank.items()}
        sel.train(training)
        np.random.seed(11)
        random.seed(12)
        return sel(labels, loc, [[1, 2, 3], [2]])

    ref = reference_outputs("host", f"query_selector_{training}_{kshot}_{text_rate}",
                            lambda: dict(zip("qmh", select(ref_loader.query_selector().QuerySelector))))
    q1, m1, h1 = select(QuerySelector)
    assert ref_equal(q1, ref["q"]) and ref_equal(m1, ref["m"]) and ref["h"] == h1
    assert set(m1.unique().tolist()) <= {0.0, 1.0}


def test_query_selector_without_bank():
    from mqdet_b200.modeling.query_selector.query_selector import QuerySelector
    assert QuerySelector(_vq_cfg())([[1]], [torch.ones(1, 4)]) == (None, None, None)


def test_boxlist_vs_reference():
    from mqdet_b200.structures.bounding_box import BoxList
    g = torch.Generator().manual_seed(3)
    xyxy = torch.rand(50, 4, generator=g) * 300 - 40
    xyxy[:, 2:] = xyxy[:, :2] + torch.rand(50, 2, generator=g) * 200 - 20     # some empty / inverted boxes
    size = (213, 160)
    idx = torch.tensor([4, 9, 30])

    def ops(cls):
        bl = cls(xyxy.clone(), size, "xyxy")
        bl.add_field("scores", torch.arange(50.0))
        bl.add_field("labels", torch.arange(50) % 7)
        out = {"area": bl.area()}
        w = bl.convert("xywh")
        out.update(xywh=w.bbox, xywh_area=w.area(), back=w.convert("xyxy").bbox, idx_bbox=bl[idx].bbox, idx_labels=bl[idx].get_field("labels"))
        c = bl.clip_to_image(remove_empty=True)
        out.update(clip_bbox=c.bbox, clip_scores=c.get_field("scores"), clipped_in_place=bl.bbox)
        return out, bl, w

    ref = reference_outputs("host", "boxlist", lambda: ops(ref_loader.bounding_box().BoxList)[0], full=("area", "xywh", "xywh_area", "back",
                            "idx_bbox", "idx_labels", "clip_bbox", "clip_scores", "clipped_in_place"))
    got, b, bw = ops(BoxList)
    assert bw.mode == "xywh" and sorted(got) == sorted(ref)
    for k in ref:                                                    # clip_to_image clips in place in both
        assert torch.equal(got[k], ref[k]), k
    assert b.copy_with_fields("scores").fields() == ["scores"] and len(b.to("cpu")) == 50
    with pytest.raises(KeyError):
        b.copy_with_fields("missing")
    with pytest.raises(ValueError):
        BoxList(torch.zeros(3, 5), size)


def test_to_image_list_vs_reference():
    from mqdet_b200.structures.image_list import to_image_list
    g = torch.Generator().manual_seed(5)
    imgs = [torch.randn(3, 50, 71, generator=g), torch.randn(3, 64, 40, generator=g), torch.randn(3, 33, 33, generator=g)]

    def compute():
        lists = [ref_loader.image_list().to_image_list(imgs, div) for div in (0, 32)]
        return {"tensors": [r.tensors for r in lists], "sizes": [[list(s) for s in r.image_sizes] for r in lists]}
    ref = reference_outputs("host", "to_image_list", compute)
    for div, rt, rs in zip((0, 32), ref["tensors"], ref["sizes"]):
        m = to_image_list(imgs, div)
        assert ref_equal(m.tensors, rt)
        assert [tuple(s) for s in rs] == [tuple(s) for s in m.image_sizes]
    one = to_image_list(imgs[0])
    assert one.tensors.shape == (1, 3, 50, 71) and one.image_sizes == [(50, 71)]
    assert to_image_list(one) is one


def test_shard_indices_cover_every_image_once():
    from mqdet_b200 import parallel
    for n, world in [(8, 1), (8, 2), (13, 4), (3, 8)]:
        seen = []
        for r in range(world):
            seen += list(parallel.shard_indices(n, r, world))
        assert sorted(seen) == list(range(n))
