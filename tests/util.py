"""Shared helpers for the parity tests."""
import math
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# north_star: "outputs match the reference's own forward on identical inputs within 1e-3 fp16 tolerance".
# Read as: max |out - ref| <= 1e-3 * max|ref| + 1e-3 per compared tensor (fp16 operands, fp32 accumulation/statistics).
FP16_TOL = 1e-3


def rel_err(out, ref):
    out = out.detach().float().cpu()
    ref = ref.detach().float().cpu()
    return (out - ref).abs().max().item() / (ref.abs().max().item() + 1e-12)


_records = []


def _dump_records():
    if _records and os.path.isdir(os.path.join(ROOT, "gpurun_out")):
        import json
        with open(os.path.join(ROOT, "gpurun_out", "parity_errors.json"), "w") as f:
            json.dump(_records, f, indent=1)


import atexit  # noqa: E402

atexit.register(_dump_records)


def assert_close(out, ref, tol=FP16_TOL, what="", defer=None):
    out = out.detach().float().cpu()
    ref = ref.detach().float().cpu()
    assert out.shape == ref.shape, f"{what}: shape {tuple(out.shape)} vs {tuple(ref.shape)}"
    assert torch.isfinite(out).all(), f"{what}: non-finite output"
    err = (out - ref).abs().max().item()
    bound = tol * ref.abs().max().item() + tol
    _records.append(dict(what=what, max_abs_err=err, bound=bound, ref_absmax=ref.abs().max().item(),
                         rel=err / (ref.abs().max().item() + 1e-12), mean_abs_err=(out - ref).abs().mean().item(),
                         ref_absmean=ref.abs().mean().item()))
    if defer is not None:
        if err > bound:
            defer.append(f"{what}: max|err| {err:.3e} > {bound:.3e}")
        return err
    assert err <= bound, f"{what}: max|err| {err:.3e} > {bound:.3e} (max|ref| {ref.abs().max().item():.3e})"
    return err


# ---- outputs of the reference's own code, stored under tests/golden/reference/ ------------------------------------------
# The pinning tests compare against what the reference's modules / kernels computed on seeded inputs.  Those runs need the
# reference sources (and, for its CUDA kernels, a GPU), so their outputs are stored: tensors of at most REF_FULL elements
# whole, larger ones as REF_SAMPLE entries at fixed positions plus max|x| and mean|x| of the whole tensor.
REFERENCE_DIR = os.path.join(ROOT, "tests", "golden", "reference")
REF_FULL, REF_SAMPLE = 1024, 256


def _sample_positions(numel):
    """Fixed positions spread over a flat tensor: a stride coprime with ``numel`` visits distinct elements."""
    stride = 2654435761 % numel or 1
    while math.gcd(stride, numel) != 1:
        stride += 1
    return torch.tensor([(i * stride + 7) % numel for i in range(min(REF_SAMPLE, numel))], dtype=torch.long)


def _condense(x, full, keep=False):
    if isinstance(x, torch.Tensor):
        x = x.detach().cpu().contiguous()
        if keep or x.numel() <= REF_FULL:
            return x.clone()
        fin = x[torch.isfinite(x)].abs().double() if x.is_floating_point() else x.abs().double()
        return {"sampled": list(x.shape), "val": x.reshape(-1)[_sample_positions(x.numel())].clone(),
                "absmax": fin.max().item() if fin.numel() else 0.0, "absmean": fin.mean().item() if fin.numel() else 0.0}
    if isinstance(x, (list, tuple)):
        return [_condense(v, full, keep) for v in x]
    if isinstance(x, dict):
        return {k: _condense(v, full, keep or k in full) for k, v in x.items()}
    return x


def reference_outputs(fixture, case, compute, full=()):
    """The stored outputs of the reference for ``case`` (tests/golden/reference/<fixture>.pt).  ``compute`` runs the reference's
    own code and returns a dict of tensors, lists of tensors and plain values; it runs only when MQDET_RECORD_REFERENCE names a
    directory, which then receives the condensed result (keys listed in ``full`` are kept whole).  Record with
    ``MQDET_RECORD_REFERENCE=tests/golden/reference python -m pytest <the test>`` where the reference can run."""
    out_dir = os.environ.get("MQDET_RECORD_REFERENCE")
    if not out_dir:
        return torch.load(os.path.join(REFERENCE_DIR, f"{fixture}.pt"))[case]
    fx = _condense(compute(), set(full))
    path = os.path.join(out_dir, f"{fixture}.pt")
    os.makedirs(out_dir, exist_ok=True)
    stored = torch.load(path) if os.path.exists(path) else {}
    stored[case] = fx
    torch.save(stored, path)
    return fx


def ref_pair(got, ref):
    """(got, ref) over the entries of the stored reference output ``ref`` (all of them when it was stored whole)."""
    got = got.detach().cpu()
    if isinstance(ref, dict):
        assert list(got.shape) == ref["sampled"], f"shape {tuple(got.shape)} vs {tuple(ref['sampled'])}"
        return got.reshape(-1)[_sample_positions(got.numel())], ref["val"]
    assert got.shape == ref.shape, f"shape {tuple(got.shape)} vs {tuple(ref.shape)}"
    return got, ref


def ref_absmax(ref):
    if isinstance(ref, dict):
        return ref["absmax"]
    fin = ref[torch.isfinite(ref)] if ref.is_floating_point() else ref
    return fin.abs().max().item() if fin.numel() else 0.0


def ref_close(got, ref, tol, what="", atol=1e-6):
    """max|got - ref| <= tol * max|finite ref| + atol over the stored entries (and the same bound on the mean of |x| when
    sampled); non-finite entries of ref must be matched exactly."""
    g, r = ref_pair(got, ref)
    fin = torch.isfinite(r)
    assert torch.equal(g[~fin], r[~fin]), f"{what}: non-finite entries differ"
    bound = tol * ref_absmax(ref) + atol
    err = (g[fin].double() - r[fin].double()).abs().max().item() if fin.any() else 0.0
    assert err <= bound, f"{what}: {err:.3e} > {bound:.3e}"
    if isinstance(ref, dict):
        am = got.detach().cpu().double()
        am = am[torch.isfinite(am)].abs().mean().item()
        assert abs(am - ref["absmean"]) <= bound, f"{what}: mean|x| {am:.6e} vs {ref['absmean']:.6e}"


def ref_equal(got, ref):
    g, r = ref_pair(got, ref)
    return torch.equal(g, r)


def vq_cfg(**over):
    """The VISION_QUERY block of configs/pretrain/mq-glip-t.yaml:132-141 as an attribute namespace (yacs is absent)."""
    vq = dict(ENABLED=True, FIX_ATTN_GATE=-1.0, CONDITION_GATE=True, NONLINEAR_GATE=True, NO_CAT=True,
              ADD_ADAPT_LAYER=False, RETURN_ATTN_GATE_VALUE=False, VISION_SCALE=1.0, AUGMENT_IMAGE_WITH_QUERY=False,
              TEXT_DROPOUT=0.4, NEW_MASK_TOKEN=False, QUERY_FUSION=False, SHARE_KV=False, NUM_QUERY_PER_CLASS=5)
    vq.update(over)
    return types.SimpleNamespace(VISION_QUERY=types.SimpleNamespace(**vq))


def load_sd(module, sd, prefix=""):
    """Load a flat {name: tensor} dict (reference state_dict names) into a module, strictly."""
    own = module.state_dict()
    sub = {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    missing = [k for k in own if k not in sub]
    extra = [k for k in sub if k not in own]
    assert not missing and not extra, f"state_dict mismatch: missing={missing[:5]} extra={extra[:5]}"
    module.load_state_dict(sub, strict=True)
    return module
