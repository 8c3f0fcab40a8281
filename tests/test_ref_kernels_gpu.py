"""GPU: pins the two 'parity unpinned' native ops against the REFERENCE's own CUDA kernels (built unmodified for sm_100a into
oracle/_ref/ by oracle/build_ref.py where the reference's sources are present); their outputs on the seeded inputs below are
stored under tests/golden/reference/ref_kernels.pt (recorded on a B200: see util.reference_outputs):
  * ml_nms — kept-index lists must be bit-identical (csrc/cuda/ml_nms.cu);
  * modulated_deform_conv_forward — including the DyConv[0] call where offsets/masks produced at a finer level are
    re-read through the coarser output's strides (vldyhead.py:212-224, deform_conv_kernel_cuda.cu:605-618)."""
import glob
import importlib.util
import os

import pytest
import torch

from util import ROOT, ref_close, reference_outputs

pytestmark = pytest.mark.gpu


def _ref():
    """The reference's compiled extension from oracle/_ref, or None where it has not been built."""
    so = glob.glob(os.path.join(ROOT, "oracle", "_ref", "mqdet_ref_C*.so"))
    if not so:
        return None
    spec = importlib.util.spec_from_file_location("mqdet_ref_C", so[0])
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("n,nlabels", [(65, 3), (1000, 10), (5000, 80)])
def test_ml_nms_equals_reference_kernel(dev, n, nlabels):
    from test_nms_gpu import _boxes
    from mqdet_b200 import ops
    from oracle import restate
    boxes, scores, labels = _boxes(900 + n, n, nlabels)
    scores = torch.unique(scores)[:n] if torch.unique(scores).numel() >= n else scores + torch.arange(n) * 1e-7
    boxes, labels = boxes[: scores.numel()], labels[: scores.numel()]  # distinct scores: ATen's sort order == stable order
    want = reference_outputs("ref_kernels", f"ml_nms_{n}_{nlabels}",
                             lambda: {"keep": _ref().ml_nms(boxes.to(dev), scores.to(dev), labels.to(dev), 0.6)}, full=("keep",))["keep"]
    got = ops.ml_nms(boxes.to(dev), scores.to(dev), labels.to(dev), 0.6).cpu()
    assert torch.equal(got, want)
    assert torch.equal(restate.ml_nms(boxes, scores, labels, 0.6), want)  # the oracle is pinned by the same kernel


def _ref_dcn(ref, x, offset, mask, weight, bias, stride):
    B, C, H, W = x.shape
    Ho, Wo = (H + 2 - 3) // stride + 1, (W + 2 - 3) // stride + 1
    out = x.new_empty(B, weight.shape[0], Ho, Wo)
    ref.modulated_deform_conv_forward(x, weight, bias, x.new_empty(0), offset, mask, out, x.new_empty(0), 3, 3, stride, stride,
                                      1, 1, 1, 1, 1, 1, True)
    return out


def test_dcnv2_equals_reference_kernel_including_quirk(dev):
    from mqdet_b200 import ops
    from mqdet_b200.modeling.rpn.vldyhead import _conv_w16
    from oracle import restate, synth
    gen = synth.Gen(31)
    sizes = [(20, 28), (10, 14), (5, 7)]
    B, C = 2, 256
    feats = [gen.randn(B, C, h, w).half().float() for h, w in sizes]  # fp16-exact inputs
    om = [gen.randn(B, 27, h, w, scale=1.5) for h, w in sizes]
    w = (gen.randn(C, C, 3, 3, scale=0.03)).half().float()
    bias = gen.randn(C, scale=0.1)
    lv = ops.Levels(sizes, dev)
    x16 = restate.flatten_levels(feats).half().to(dev).contiguous()
    om_flat = torch.zeros(B, lv.N, 32)
    om_flat[:, :, :27] = restate.flatten_levels(om)
    om_dev = om_flat.to(dev).contiguous()
    wparam = torch.nn.Parameter(w.to(dev))
    cases = [(branch, stride, l) for branch, stride in ((1, 1), (2, 2), (0, 1)) for l in range(len(sizes)) if branch == 1 or l > 0]

    def inputs(branch, l):
        if branch == 1:
            return feats[l], l
        if branch == 2:
            return feats[l - 1], l
        return feats[l], l - 1  # conv on level l with the offsets of the finer level l-1 (the quirk)

    def compute():
        ref, out = _ref(), {}
        for branch, stride, l in cases:
            xin, lo = inputs(branch, l)
            off = om[lo][:, :18].contiguous().to(dev)
            msk = om[lo][:, 18:].sigmoid().contiguous().to(dev)
            out[f"{branch}_{l}"] = _ref_dcn(ref, xin.to(dev), off, msk, w.to(dev), bias.to(dev), stride)
        return out
    wants = reference_outputs("ref_kernels", "dcnv2", compute)
    for branch, stride in ((1, 1), (2, 2), (0, 1)):
        cols = ops.dcn_cols(x16, om_dev, lv, branch)
        y = ops.gemm(cols, _conv_w16(wparam), bias=bias.to(dev), out_dtype=torch.float32)
        rows = lv.N if branch == 1 else lv.N1
        y = y.view(B, rows, C).cpu()
        o = 0
        for l in range(len(sizes)):
            if (branch, stride, l) not in cases:
                continue
            xin, lo = inputs(branch, l)
            want = wants[f"{branch}_{l}"]
            h, wd = sizes[l]
            got = y[:, o:o + h * wd].transpose(1, 2).reshape(B, C, h, wd)
            assert torch.isfinite(got).all(), f"DCNv2 branch {branch} level {l}: non-finite output"
            ref_close(got, want, 1e-3, f"DCNv2 branch {branch} level {l} vs reference kernel", atol=1e-3)
            orc = restate.dcn_v2(xin, om[lo][:, :18].reshape(B, -1), om[lo][:, 18:].sigmoid().reshape(B, -1), w, bias, stride)
            ref_close(orc, want, 1e-5, f"oracle dcn_v2 branch {branch} level {l} vs reference kernel", atol=1e-5)
            o += h * wd
