#!/usr/bin/env python
"""bench.py — images/sec of the MQ-GLIP-T multi-modal query forward on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl mqdet|reference] [--dump-outputs DIR]

A step = one forward of ``GeneralizedVLRCNN_New`` (Swin-T -> FPN -> QuerySelector/PreSelect/GCP-BERT -> 6x[BiAttention,
BERT layer, DyConv] -> dot-product token head -> ATSS post-processing + ml_nms) over one batch of synthetic 800x1333
images (zero-padded to 800x1344), an 80-class COCO-shaped prompt (T = 256 tokens) and K = 5 vision queries per class,
random-init weights of the real architecture (no checkpoints offline).

  value : images/s with the batch already resident in HBM (CUDA-event time of K steps, max over ranks).
  e2e   : the same metric through the public API with HOST buffers: every step copies its images from pinned host
          memory, runs the forward and reads the fixed-shape detections back.
  N > 1 : one process per GPU (torchrun), images sharded over ranks (weak scaling, B per GPU fixed), ONE NCCL all-gather
          of the fixed-shape per-image detections per step.
  --impl reference : the CPU oracle (oracle/restate.py — the reference's algorithm restated; its own modules cannot run
          the full forward on CPU, SURVEY.md §8c) on the host cores, one image per step (bounded sample), rank 0 only.
  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned as DIR/<name>.npy (float32):
          inputs and weights come from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec MQ-GLIP-T 800x1333, 5 vis-queries, 80-class prompt"
H_IMG, W_IMG, NCLS, KQ = 800, 1333, 80, 5


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "tflops": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "src": "measured (MEASURED_PEAKS.json, sustained)"}
    return {"hbm_gbs": 6650.0, "tflops": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def cpu_threads():
    """Host threads for the CPU oracle: all cores up to 32.  Beyond that the restatement (many small tensor ops between the
    large matmuls) gets slower, not faster: measured 16.6 s / image on 8 threads vs 97.7 s / image on 128 threads."""
    return max(1, min(os.cpu_count() or 1, int(os.environ.get("MQDET_CPU_THREADS", "32"))))


class ClockSampler:
    """nvidia-smi clocks / power / throttle reasons of every GPU of the job, sampled DURING the timed region (rank 0 polls)."""

    def __init__(self, idx):
        self.idx = list(idx) if isinstance(idx, (list, tuple, range)) else [idx]
        self.rows, self.proc = [], None

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", ",".join(str(i) for i in self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 8 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        per_gpu = []
        for g in sorted({r[0] for r in rows}):
            sm = sorted(int(r[1]) for r in rows if r[0] == g)
            pw = sorted(float(r[3]) for r in rows if r[0] == g and r[3].replace(".", "", 1).isdigit())
            per_gpu.append({"gpu": int(g), "sm_mhz": sm[len(sm) // 2], "power_w": pw[len(pw) // 2] if pw else None})
        sm_all = sorted(int(r[1]) for r in rows)
        mx = [int(r[2]) for r in rows if r[2].isdigit()]
        # sm_mhz = the LOWEST per-GPU median under load (the slowest GPU paces a max-over-ranks number)
        return {"sm_mhz": min(g["sm_mhz"] for g in per_gpu) if per_gpu else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm_all), "per_gpu": per_gpu}


def traffic_note():
    """(dram bytes per launch of the dominant kernel from the committed ncu --set full capture, its source) or (None, why)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("dram_bytes_per_launch"), d.get("source")
    return None, "no ncu --set full capture summarised in profiles/r02_traffic.json"


# Algorithmic work per IMAGE and stage (SURVEY.md §8d, 80-class prompt, fp16 storage): (GFLOP, activation MB per image that
# must cross HBM at least once, weight MB read once per step)
STAGE_WORK = {
    "swin": (96.0, 2 * 12.9 * 12, 55.0), "fpn": (28.0, 2 * 11.5, 7.0),
    "preselect": (12.2, 2.86 + 0.8, 12.2), "gcp x6": (21.6, 6 * (0.79 + 0.61), 79.1),
    "bert layers x18": (45.9 + 6 * 3.83, 18 * 0.79, 18 * 14.2),
    "fusion x6 (biattention)": (860.1, 6 * (22.9 + 0.79), 6 * 12.6), "dyconv x6": (254.5, 6 * 3 * 23.0, 6 * 3.6),
    "dot-product head": (2.94, 11.47 + 0.13 + 11.47, 0.4), "post-processing (atss + ml_nms)": (0.025, 11.5 + 0.36 + 3.2, 0.0),
}


def stage_profile(model, eager_step, B, pk):
    """CUDA-event time of every stage of ONE eager forward + its algorithmic FLOPs / bytes (STAGE_WORK) -> per stage
    {ms, tensor_frac, hbm_frac}: the north-star asks for both fractions on the GCP + fusion path."""
    import torch
    from mqdet_b200 import ops
    import mqdet_b200.modeling.language_backbone.modeling_bert_new as mb
    events, undo = [], []

    def wrap(obj, name, label):
        fn = getattr(obj, name)

        def w(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **k)
            e1.record()
            events.append((label, e0, e1))
            return r
        setattr(obj, name, w)
        undo.append((obj, name, fn))

    lm = model.language_backbone.body.model
    wrap(model.backbone.body, "forward_flat", "swin")
    wrap(model.backbone.fpn, "forward_flat", "fpn")
    wrap(lm.pre_select, "forward", "preselect")
    for blk in lm.encoder.qv_layer:
        wrap(blk, "forward", "gcp x6")
    wrap(mb.BertLayer, "forward", "bert layers x18")
    tower = model.rpn.head.dyhead_tower
    for i in range(0, len(tower), 3):
        wrap(tower[i].b_attn, "forward_flat", "fusion x6 (biattention)")
        wrap(tower[i + 2], "forward_flat", "dyconv x6")
    wrap(ops, "atss_postprocess", "post-processing (atss + ml_nms)")
    wrap(ops, "l2_normalize", "_head_start")
    overlap, overlap_p = model.rpn.head.overlap_text_stream, model.overlap_text_prefix
    model.rpn.head.overlap_text_stream = False  # stage times are taken with the two tower branches one after the other
    model.overlap_text_prefix = False           # ... and the BERT prefix after the visual backbone, not next to it
    try:
        for _ in range(2):
            events.clear()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            eager_step()
            t1.record()
            torch.cuda.synchronize()
    finally:
        model.rpn.head.overlap_text_stream = overlap
        model.overlap_text_prefix = overlap_p
        for obj, name, fn in reversed(undo):
            setattr(obj, name, fn)
    agg = {}
    for label, a, b in events:
        agg[label] = agg.get(label, 0.0) + a.elapsed_time(b)
    # dot-product head = from l2_normalize to the start of the post-processing
    hs = [a for lb, a, _ in events if lb == "_head_start"]
    ps = [a for lb, a, _ in events if lb.startswith("post-processing")]
    agg.pop("_head_start", None)
    if hs and ps:
        agg["dot-product head"] = hs[0].elapsed_time(ps[0])
    out = {"eager_step_ms": t0.elapsed_time(t1)}
    for label, ms_ in agg.items():
        gf, act_mb, w_mb = STAGE_WORK[label]
        flops, byts = gf * 1e9 * B, (act_mb * B + w_mb) * 1e6
        out[label] = {"ms": round(ms_, 3), "algorithmic_gflop": round(flops / 1e9, 1), "algorithmic_mb": round(byts / 1e6, 1),
                      "tensor_frac": round(flops / (ms_ / 1e3) / 1e12 / pk["tflops"], 4),
                      "hbm_frac": round(byts / (ms_ / 1e3) / 1e9 / pk["hbm_gbs"], 4)}
    return out


def run_lvis(args):
    """BASELINE config 3: MQ-GLIP-L (Swin-L window 12, 8 fusion layers), batch 4 / GPU, LVIS-shaped vocabulary of 1203 classes
    evaluated as 31 prompts of 40 classes (TEST.CHUNKED_EVALUATION 40), K = 5 queries per class, 300 detections per chunk.
    A step = ALL chunks of one image batch: Swin-L + FPN once, the chunks batched through the language backbone / fusion
    tower / post-processing (mqdet_b200 forward_chunked_device); N > 1: the chunks shard over ranks (chunk c -> rank c % N,
    strong scaling of the step) and ONE all-gather returns every chunk's packed detections."""
    import torch
    import torch.distributed as dist
    from mqdet_b200 import _lib, ops, parallel
    from mqdet_b200.config import mq_glip_l_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.structures.image_list import ImageList
    from tools import synth
    _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    B, NCLS_L, CHUNK = (args.batch if args.batch != 8 else 4), 1203, 40
    gen = synth.Gen(1237)
    chunks = synth.chunked_prompts(NCLS_L, CHUNK, 256, gen)
    bank = {}
    for _, _, pm in chunks:
        bank.update(synth.query_bank(pm, KQ, gen))
    img = synth.images(gen, B, H_IMG, W_IMG)
    sd = synth.detector_sd(synth.Gen(98), num_convs=8, bias0=args.bias0,
                           swin=dict(depths=(2, 2, 18, 2), heads=(6, 12, 24, 48), embed=192, ws=12))
    model = GeneralizedVLRCNN_New(mq_glip_l_cfg())
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            sd[k] = v
    model.load_state_dict(sd, strict=True)
    del sd
    model = model.to(dev).eval()
    model.query_selector.set_query_bank(bank)
    caps = [{"input_ids": i, "attention_mask": a} for i, a, _ in chunks]
    pmaps = [pm for _, _, pm in chunks]
    mine = parallel.shard_chunks(len(chunks), rank, world)
    il = ImageList(img.to(dev), [(H_IMG, W_IMG)] * B)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def step():
        out = model.forward_chunked_device(il, caps, pmaps, chunks_per_pass=args.chunks_per_pass, chunk_ids=mine)
        return parallel.all_gather_chunks(out["det_packed"], len(chunks))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, args.warmup)):
        res = step()
    barrier()
    ops.launch_count = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    clocks = ClockSampler(range(world))
    if rank == 0:
        clocks.start()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        res = step()
        ev[i][1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"detections": res})  # [chunks, B, max_out + 1, 6]: boxes, score, label; count row last
    clk = clocks.stop() if rank == 0 else None
    ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    t = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    if rank == 0:
        nd = res[:, :, -1, 0].sum().item()
        print(json.dumps({
            "metric": "images/sec MQ-GLIP-L 800x1333, LVIS 1203-class chunked prompt (31 x 40 classes), 5 vis-queries", "value": B / (ms / 1e3),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"MQ-GLIP-L (Swin-L w12 + FPN once per image, 31 prompt chunks batched {args.chunks_per_pass} per pass through "
                                   f"BERT+GCP, 8x fusion/DyConv, head, ATSS+ml_nms 300/chunk), batch {B}, BASELINE config 3, random-init weights",
                       "global_batch": B, "parallelism": f"prompt chunks sharded over {world} rank(s), 1 NCCL all-gather of [chunks,B,{model.max_out() + 1},6]",
                       "chunk_forwards_per_step": B * len(chunks), "detections_returned_per_step": nd,
                       "l2": "256 MiB buffer written between timed steps"},
            "gpu_launches": ops.launch_count, "clocks": clk}), flush=True)
    finish(world)


def run_gdino(args):
    """BASELINE config 4: MQ-GroundingDINO-T (Swin-T, 4 levels, 6 encoder [fusion + text enhancer + deformable] + 6 decoder layers,
    900 queries, two-stage), batch 2 / GPU (16 over 8 GPUs), ODinW-13-shaped 13-class prompt, K = 5 vision queries per class.
    A step = one forward of ``GroundingDINO`` over the local images -> packed detections; N > 1: images shard over ranks (weak
    scaling) and ONE NCCL all-gather returns the fixed-shape detections [B, 901, 6] of every rank."""
    import torch
    import torch.distributed as dist
    from mqdet_b200 import _lib, ops, parallel
    from mqdet_b200.config import mq_groundingdino_t_cfg
    from mqdet_b200.modeling.groundingdino.groundingdino import GroundingDINO
    from mqdet_b200.structures.image_list import ImageList
    from tools import synth
    _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    B = args.batch if args.batch != 8 else 2
    gen = synth.Gen(1238 + rank)
    ids, am, pmap = synth.prompt(13, 2, 256, gen)
    bank = synth.query_bank(pmap, KQ, gen)
    img = synth.rgb_images(gen, B, H_IMG, W_IMG)
    sd = synth.gdino_sd(synth.Gen(99))
    model = GroundingDINO(mq_groundingdino_t_cfg())
    for k, v in model.state_dict().items():
        if k.endswith("relative_position_index"):
            sd[k] = v
    model.load_state_dict(sd, strict=True)
    del sd
    model = model.to(dev).eval()
    model.query_selector.set_query_bank(bank)
    caps = {"input_ids": ids, "attention_mask": am}
    il = ImageList(img.to(dev), [(H_IMG, W_IMG)] * B)
    host = img.pin_memory()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    # the public API: mqdet_b200.engine.inference.GroundingDINOEngine — the forward has a fixed shape and no host synchronisation once
    # the prompt / geometry state is cached, so it is captured as ONE CUDA graph over a static input buffer (--no-graph: ~780 eager
    # launches per step, launch-bound at 2 images) and replayed per batch; N > 1: one all-gather of the packed result per step
    from mqdet_b200.engine.inference import GroundingDINOEngine
    engine = GroundingDINOEngine(model, caps, pmap, tuple(img.shape), [(H_IMG, W_IMG)] * B, use_graph=not args.no_graph)
    graph, graph_note = engine.graph, engine.note
    engine.static_in.copy_(il.tensors)

    def step(x=None):
        return engine.step_device(x)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(3, args.warmup)):
        res = step()
    barrier()
    ops.launch_count = 0
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    clocks = ClockSampler(range(world))
    if rank == 0:
        clocks.start()
    for i in range(args.steps):
        flush.zero_()
        ev[i][0].record()
        res = step()
        ev[i][1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"detections": res})  # [world * B, num_queries + 1, 6]: boxes, score, label; count row last
    launches = ops.launch_count
    if graph is not None:  # launches replayed per step = the launches recorded while capturing
        ops.launch_count = 0
        model.forward_device(il, caps, pmap)
        launches = ops.launch_count * args.steps
    clk = clocks.stop() if rank == 0 else None
    ms = sum(a.elapsed_time(b) for a, b in ev) / args.steps
    # end to end through the public API with HOST buffers: pinned images -> H2D -> forward -> packed detections -> D2H -> BoxLists
    barrier()
    t0 = time.time()
    nd = 0
    for boxlists in engine.run([host] * args.steps):   # pinned host -> input buffer -> replay (-> all-gather) -> D2H -> list[BoxList]
        nd += sum(len(b) for b in boxlists)
    barrier()
    e2e_ms = (time.time() - t0) * 1e3 / args.steps
    t = torch.tensor([ms, e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, e2e_ms = float(t[0].item()), float(t[1].item())
    if rank == 0:
        print(json.dumps({
            "metric": "images/sec MQ-GroundingDINO-T 800x1333, 13-class prompt, 5 vis-queries", "value": world * B / (ms / 1e3),
            "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"MQ-GroundingDINO-T full forward (Swin-T, input_proj+GroupNorm, BERT+GCP+PreSelect with per-category "
                                   f"text masks, 6x[BiAttention fusion, text enhancer, deformable encoder layer], two-stage top-900, "
                                   f"6 decoder layers, ContrastiveEmbed + box refinement, detections), batch {B}/GPU, 800x1333 (padded "
                                   f"800x1344), 13-class prompt T=256, K=5 (BASELINE config 4), random-init weights",
                       "global_batch": world * B, "parallelism": f"image-sharded dp{world}, 1 NCCL all-gather of [{world},{B},901,6] per step",
                       "launch": graph_note, "l2": "256 MiB buffer written between timed steps",
                       "tokenisation": "pre-tokenised ids (no bert-base-uncased vocabulary offline)"},
            "e2e": {"value": world * B / (e2e_ms / 1e3), "unit": "images/s", "h2d_bytes_per_step": int(img.numel() * 4),
                    "d2h_bytes_per_step": int(B * 901 * 6 * 4), "detections_per_step": nd / args.steps,
                    "api": "mqdet_b200.engine.inference.GroundingDINOEngine.run(host batches) -> list[BoxList] per batch",
                    "timing": "host wall clock around K steps incl. H2D, forward, D2H, BoxList construction"},
            "gpu_launches": launches, "clocks": clk}), flush=True)
    finish(world)


def init_nccl(dev):
    """One small collective per step (24.8 KB per rank): a single NCCL CTA is plenty, and every further CTA that sits on an
    SM waiting for a peer would take that SM away from the persistent one-CTA-per-SM kernels of the forward running next to
    it on the main stream.  Explicit NCCL_* settings in the environment win."""
    import torch.distributed as dist
    os.environ.setdefault("NCCL_MAX_CTAS", "1")
    os.environ.setdefault("NCCL_MIN_CTAS", "1")
    dist.init_process_group("nccl", device_id=dev)
    # ... and the persistent kernels leave that one SM to it (before any launch / graph capture): an NCCL CTA that waits for a
    # peer (ranks drift by up to a step) otherwise delays one CTA of every persistent kernel it overlaps with
    from mqdet_b200 import _lib
    _lib.check(_lib.load().mqdet_reserve_sms(int(os.environ.get("MQDET_RESERVED_SMS", "1"))), "reserve_sms")


def finish(world):
    """Leave the process group; the JSON line is already out, so a teardown that does not return within 30 s (seen with
    communicators that recorded graph-captured collectives) ends the process instead of hanging the launcher."""
    if world <= 1:
        return
    import threading
    import torch.distributed as dist
    sys.stdout.flush()
    guard = threading.Timer(30.0, lambda: os._exit(0))
    guard.daemon = True
    guard.start()
    dist.barrier()
    dist.destroy_process_group()
    guard.cancel()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)  # nothing left to finalise; interpreter teardown with NCCL/graph state alive is the other place this can hang


DUMP_MAX_ELEMENTS = 1 << 21  # per array (8 MB of float32): larger outputs are written as a fixed, seeded sample of their entries


def dump_outputs(out_dir, arrays):
    """{name: device tensor} -> out_dir/<name>.npy as float32.  An array of more than DUMP_MAX_ELEMENTS entries is written as the
    entries at DUMP_MAX_ELEMENTS flat positions drawn from a generator seeded with 0 (the same positions for the same shape)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        x = t.detach().float()
        if x.numel() > DUMP_MAX_ELEMENTS:
            idx = torch.randint(x.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
            x = x.reshape(-1)[idx.to(x.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), x.cpu().numpy())


def build_inputs(B, seed):
    import torch
    from tools import synth  # synthetic weights/inputs generator (not the measured path)
    gen = synth.Gen(seed)
    ids, am, pmap = synth.prompt(NCLS, 2, 256, gen)
    bank = synth.query_bank(pmap, KQ, gen)
    img = synth.images(gen, B, H_IMG, W_IMG)
    return gen, ids, am, pmap, bank, img


def run_reference(args):
    """CPU arm: the oracle restatement of the reference forward on the host cores, one image per step."""
    import torch
    from oracle import restate
    from tools import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_threads()
    torch.set_num_threads(cores)
    gen = synth.Gen(1235)
    sd = synth.detector_sd(gen, bias0=args.bias0)
    ids, am, pmap = synth.prompt(NCLS, 2, 256, gen)
    bank = synth.query_bank(pmap, KQ, gen)
    img = synth.images(gen, 1, H_IMG, W_IMG)
    times = []
    with torch.no_grad():
        for i in range(args.warmup + args.steps):
            t = time.time()
            restate.detector(img, (H_IMG, W_IMG), ids, am, pmap, bank, sd, K=KQ, num_classes=NCLS)
            if i >= args.warmup:
                times.append(time.time() - t)
    ms = 1e3 * sum(times) / len(times)
    v = 1e3 / ms
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "MQ-GLIP-T full forward, 1 image 800x1333 (padded 800x1344) per step, 80-class prompt, K=5"},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} step(s) of 1 image, oracle/restate.py (fp32, torch CPU, {cores} threads)"},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8, help="images per GPU per step (BASELINE config 2: 8)")
    ap.add_argument("--impl", default="mqdet", choices=["mqdet", "reference"])
    ap.add_argument("--bias0", type=float, default=-math.log((1 - 0.01) / 0.01),
                    help="dot-product head bias0 of the synthetic weights; default = the reference's own initialisation "
                         "-log((1-p)/p), PRIOR_PROB p = 0.01 (vldyhead.py:688-719, defaults.py:442).  It sets the fraction of "
                         "(location, class) pairs above the 0.05 pre-NMS threshold; the candidate / detection counts it "
                         "yields are reported in config.postprocess (-1.5 is a denser stress point: every level hits top-k)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the kernels eagerly instead of replaying the captured CUDA graph")
    ap.add_argument("--gather-every", type=int, default=8, help="steps whose packed results one all-gather exchanges (N > 1)")
    ap.add_argument("--cpu-baseline-steps", type=int, default=1)
    ap.add_argument("--config", default="coco", choices=["coco", "lvis", "gdino"],
                    help="coco: BASELINE config 2 (the headline metric); lvis: BASELINE config 3 (MQ-GLIP-L, chunked 1203-class prompt); "
                         "gdino: BASELINE config 4 (MQ-GroundingDINO-T, 2 images / GPU, 13-class prompt)")
    ap.add_argument("--chunks-per-pass", type=int, default=4)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32; large arrays as a fixed, seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the CUDA path (--impl mqdet)")
    if args.impl == "reference":
        return run_reference(args)
    if args.config == "lvis":
        return run_lvis(args)
    if args.config == "gdino":
        return run_gdino(args)

    import torch
    import torch.distributed as dist
    from mqdet_b200 import _lib, ops
    from mqdet_b200.config import mq_glip_t_cfg
    from mqdet_b200.modeling.detector.generalized_vl_rcnn_new import GeneralizedVLRCNN_New
    from mqdet_b200.structures.image_list import ImageList
    from tools import synth

    _lib.load()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        init_nccl(dev)
    B = args.batch
    gen, ids, am, pmap, bank, img = build_inputs(B, 1235 + rank)
    sd = synth.detector_sd(synth.Gen(99), bias0=args.bias0)
    model = GeneralizedVLRCNN_New(mq_glip_t_cfg())
    own = model.state_dict()
    for k in own:
        if k.endswith("relative_position_index"):
            sd[k] = own[k]
    model.load_state_dict(sd, strict=True)
    del sd
    model = model.to(dev).eval()
    model.query_selector.set_query_bank(bank)
    caps = {"input_ids": ids, "attention_mask": am}
    sizes = [(H_IMG, W_IMG)] * B
    img_host = img.pin_memory()
    img_dev = img.to(dev)
    from mqdet_b200.engine.inference import InferenceEngine
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # one eager forward: counts the kernels of a step (the graph replays exactly these) and fills every cache
    ops.launch_count = 0
    model.forward_device(ImageList(img_dev, sizes), caps, pmap)
    torch.cuda.synchronize()
    launches_per_step = ops.launch_count
    # The public inference API: the forward + the ONE collective captured as a CUDA graph, replayed per batch
    # (mqdet_b200/engine/inference.py; --no-graph runs the same calls eagerly)
    graph_note = "cuda-graph replay"
    try:
        engine = InferenceEngine(model, caps, pmap, tuple(img.shape), sizes, use_graph=not args.no_graph, warmup=max(1, args.warmup // 2),
                                 gather_every=args.gather_every)
    except Exception as e:  # noqa: BLE001 - e.g. a collective that cannot be captured on this stack: fall back to eager launches
        if args.no_graph:
            raise
        graph_note = f"eager (graph capture failed: {type(e).__name__}: {str(e)[:120]})"
        torch.cuda.synchronize()
        engine = InferenceEngine(model, caps, pmap, tuple(img.shape), sizes, use_graph=False, warmup=1, gather_every=args.gather_every)
    if args.no_graph:
        graph_note = "eager launches (--no-graph)"
    engine.stage[0].copy_(img_dev)
    engine.stage[1].copy_(img_dev)

    # ---- device-resident throughput ---------------------------------------------------------------------------------
    for i in range(args.warmup):
        engine.device_step(k=i & 1)
    barrier()
    clocks = ClockSampler(range(world))  # rank 0 polls every GPU of the job (local ranks 0..N-1 on the one node)
    if rank == 0:
        clocks.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    main_stream = torch.cuda.current_stream()
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (outside the per-step events)
        ev[i][0].record()
        engine.device_step(k=i & 1)
        ev[i][1].record()
    # the exchange ring (one all-gather per `gather_every` steps) runs on the engine's result stream behind the forward; a
    # step's bracket holds the wait for the result work issued two steps earlier, and this last bracket the flush of the ring
    # and whatever is still in flight: every collective is timed
    tail = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    tail[0].record()
    engine.flush()  # a partly filled exchange ring is gathered inside the timed region
    for e in engine.res_done + [engine.gather_done]:
        main_stream.wait_event(e)
    tail[1].record()
    barrier()
    if args.dump_outputs and rank == 0:
        # the last timed step: the packed detections InferenceEngine.run turns into BoxLists, and the head outputs they come from
        last = engine.outs[(args.steps - 1) & 1]
        dump_outputs(args.dump_outputs, {"detections": last["packed"], "dot_product_logits": last["raw"]["head"]["dot_product_logits"],
                                         "reg_ctr": last["raw"]["head"]["reg_ctr"], "fused_language": last["raw"]["head"]["hidden"]})
    launches = launches_per_step * args.steps
    ms = (sum(a.elapsed_time(b) for a, b in ev) + tail[0].elapsed_time(tail[1])) / args.steps
    t = torch.tensor([ms], device=dev)
    ms_per_rank = [ms]
    if world > 1:
        allms = torch.empty((world,), device=dev)
        dist.all_gather_into_tensor(allms, t)
        ms_per_rank = [float(x) for x in allms.tolist()]   # reported: tells a slow GPU from a systematic N > 1 cost
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = world * B / (ms / 1e3)

    # ---- end to end through the public API with host buffers ----------------------------------------------------------
    # `for boxlists in engine.run(batches)`: every batch starts in pinned HOST memory and ends as list[BoxList] built from the
    # pinned host copy of the packed result — H2D (103 MB), forward, all-gather, D2H and BoxList construction all inside the
    # timed region.  The engine uploads batch s+1 on a copy stream while batch s computes (a prefetching data loader).
    for _ in engine.run([img_host] * 2):
        pass
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_boxes = 0
    t_wall = time.time()
    e0.record()
    for boxlists in engine.run([img_host] * args.steps):
        n_boxes += sum(len(bl) for bl in boxlists)
    torch.cuda.current_stream().wait_event(engine.gather_done)  # the run's last exchange (flush) is inside the timed region
    e1.record()
    barrier()
    e2e_wall_ms = 1e3 * (time.time() - t_wall) / args.steps
    e2e_ms = max(e0.elapsed_time(e1) / args.steps, 0.0)
    t = torch.tensor([e2e_ms], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    clk = clocks.stop() if rank == 0 else None
    # operating point of the post-processing (what the synthetic weights make it do), from the last step's device counters
    o = engine.outs[0]["raw"] if engine.use_graph else model.forward_device(ImageList(img_dev, sizes), caps, pmap)
    pp = {"bias0": args.bias0, "pre_nms_thresh": 0.05,
          "pre_nms_boxes_per_image_after_topk": float(o["cand_totals"].float().mean().item()),
          "detections_per_image": float(o["num"].float().mean().item())}

    # ---- roofline of the dominant kernel family (the tcgen05 GEMM): every launch timed with CUDA events on its stream ----
    def eager_step():
        return model.forward_device(ImageList(img_dev, sizes), caps, pmap)

    # (every stream overlap off: a kernel is timed alone on the device, not next to the other branch)
    ov_t, ov_p = model.rpn.head.overlap_text_stream, model.overlap_text_prefix
    model.rpn.head.overlap_text_stream = model.overlap_text_prefix = False
    prof = ops.GEMM_PROFILE = []
    kprof = ops.KERNEL_PROFILE = []
    eager_step()
    torch.cuda.synchronize()
    ops.GEMM_PROFILE = None
    ops.KERNEL_PROFILE = None
    model.rpn.head.overlap_text_stream, model.overlap_text_prefix = ov_t, ov_p
    g_ms = sum(a.elapsed_time(b) for a, b, _, _ in prof)
    g_flops = sum(f for _, _, f, _ in prof)
    pk = peaks()
    achieved = g_flops / (g_ms / 1e3) / 1e12 if g_ms > 0 else 0.0
    # per tensor-core kernel: measured time against the roofline time of each launch, max(flops / tensor peak, bytes / HBM
    # peak) with ALGORITHMIC flops and bytes — the family of GEMMs mixes tensor-bound and HBM-bound shapes, so one ratio against
    # one peak misstates it
    tc_ms = sum(k[0].elapsed_time(k[1]) for k in kprof)
    tc_flops = sum(k[3] for k in kprof)
    tc_executed = sum(k[5] for k in kprof)
    tc_achieved = tc_flops / (tc_ms / 1e3) / 1e12 if tc_ms > 0 else 0.0
    kern = {}
    for e0, e1, name, fl, by, ex in kprof:
        t = e0.elapsed_time(e1)
        k = kern.setdefault(name, {"launches": 0, "ms": 0.0, "flops": 0.0, "executed": 0.0, "bytes": 0.0, "roof_ms": 0.0, "hbm_bound_ms": 0.0})
        # roofline time of a launch from what it EXECUTES on the tensor cores (<= the algorithmic count where projections are folded
        # algebraically), so no fraction can exceed 1; the algorithmic rate is reported next to it
        t_tensor, t_hbm = ex / (pk["tflops"] * 1e12) * 1e3, by / (pk["hbm_gbs"] * 1e9) * 1e3
        k["launches"] += 1
        k["ms"] += t
        k["flops"] += fl
        k["executed"] += ex
        k["bytes"] += by
        k["roof_ms"] += max(t_tensor, t_hbm)
        if t_hbm > t_tensor:
            k["hbm_bound_ms"] += t
    kernels = []
    for name, k in sorted(kern.items(), key=lambda kv: -kv[1]["ms"]):
        kernels.append({"kernel": name, "launches": k["launches"], "ms_per_step": round(k["ms"], 3),
                        "algorithmic_tflops": round(k["flops"] / (k["ms"] / 1e3) / 1e12, 1),
                        "algorithmic_gbs": round(k["bytes"] / (k["ms"] / 1e3) / 1e9, 1),
                        "executed_tflops": round(k["executed"] / (k["ms"] / 1e3) / 1e12, 1),
                        "tensor_frac": round(k["executed"] / (k["ms"] / 1e3) / 1e12 / pk["tflops"], 3),
                        "roofline_frac": round(k["roof_ms"] / k["ms"], 3),
                        "ms_in_hbm_bound_launches": round(k["hbm_bound_ms"], 3)})
    stages = stage_profile(model, eager_step, B, pk) if rank == 0 else None

    if rank == 0:
        res = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"MQ-GLIP-T full forward (Swin-T+FPN, BERT+GCP+PreSelect, 6x fusion/DyConv, dot-product "
                                   f"head, ATSS+ml_nms), batch {B}/GPU, 800x1333 (padded 800x1344), 80-class prompt T=256, "
                                   f"K=5 queries/class (BASELINE config 2), random-init weights",
                       "global_batch": world * B, "parallelism": f"image-sharded dp{world}, 1 NCCL all-gather of [{engine.G},B,{model.max_out() + 1},6] (detections + count row) per {engine.G} steps (+ flush)",
                       "launch": graph_note + ("; tower text branch on a second stream" if model.rpn.head.overlap_text_stream else ""),
                       "l2": "256 MiB buffer written between timed steps", "postprocess": pp,
                       "tokenisation": "pre-tokenised ids (no bert-base-uncased vocabulary offline); prompt state cached per prompt"},
            # the dominant kernel family = the tcgen05 kernels: every matrix product of the step (the set round 1 ran through
            # the one GEMM kernel; since round 2 the attention products and the DCNv2 convolutions have kernels of their own)
            "roofline": {"bound": "tensor", "achieved": tc_achieved, "peak": pk["tflops"], "unit": "TFLOP/s",
                         "frac": tc_achieved / pk["tflops"], "traffic": traffic_note()[0], "peak_source": pk["src"],
                         "kernel": "tcgen05 kernels: gemm_tcp_kernel (all shapes), dcn_conv_kernel, biattn_image_kernel, "
                                   "biattn_text_kernel — every matrix product of one step", "launches": len(kprof),
                         "kernel_ms_per_step": tc_ms, "kernel_share_of_step": tc_ms / stages["eager_step_ms"] if stages else None,
                         "algorithmic_tflop_per_step": tc_flops / 1e12, "executed_tflop_per_step": tc_executed / 1e12,
                         "executed_frac": tc_executed / (tc_ms / 1e3) / 1e12 / pk["tflops"] if tc_ms > 0 else None,
                         "traffic_source": traffic_note()[1],
                         "gemm_only": {"achieved": achieved, "frac": achieved / pk["tflops"], "launches": len(prof),
                                       "kernel_ms_per_step": g_ms, "algorithmic_tflop_per_step": g_flops / 1e12},
                         "kernels": kernels, "kernels_note": "per tensor-core kernel, CUDA events around every launch of one eager "
                                                             "step: roofline_frac = sum over launches of max(EXECUTED flops / "
                                                             "tensor peak, algorithmic bytes / HBM peak) / measured time; algorithmic_tflops "
                                                             "counts the reference's arithmetic for the same work (the attention kernels fold "
                                                             "the query / value / output projections into small text-side operands, so they "
                                                             "execute less than that)",
                         "stages": stages},
            "e2e": {"value": world * B / (e2e_ms / 1e3), "unit": "images/s", "ms_per_step": e2e_ms, "wall_ms_per_step": e2e_wall_ms,
                    "h2d_bytes_per_step": img_host.numel() * 4, "d2h_bytes_per_step": engine.host[0].numel() * 4 + (engine.gathered_host.numel() * 4 // engine.G if world > 1 else 0),
                    "api": "mqdet_b200.engine.inference.InferenceEngine.run(host batches) -> list[BoxList] per batch",
                    "boxes_returned": n_boxes},
            "gpu_launches": launches, "clocks": clk, "ms_per_step_per_rank": ms_per_rank,
        }
        if not args.no_cpu_baseline and world == 1:
            import torch as _t
            from oracle import restate
            cores = cpu_threads()
            _t.set_num_threads(cores)
            g2 = synth.Gen(1235)
            sd_c = synth.detector_sd(g2, bias0=args.bias0)
            i1, a1, pm1 = synth.prompt(NCLS, 2, 256, g2)
            bk = synth.query_bank(pm1, KQ, g2)
            im1 = synth.images(g2, 1, H_IMG, W_IMG)
            ts = []
            with _t.no_grad():
                for _ in range(args.cpu_baseline_steps):
                    t0 = time.time()
                    restate.detector(im1, (H_IMG, W_IMG), i1, a1, pm1, bk, sd_c, K=KQ, num_classes=NCLS)
                    ts.append(time.time() - t0)
            res["cpu_baseline"] = {"value": 1.0 / (sum(ts) / len(ts)), "unit": "images/s", "cores": cores, "kind": "port",
                                   "sample": f"{len(ts)} forward(s) of ONE 800x1333 image, 80-class prompt, oracle/restate.py "
                                             f"fp32 on {cores} host threads"}
        print(json.dumps(res), flush=True)
    engine.close()  # captured NCCL all-gathers must be gone before the communicator is
    finish(world)


if __name__ == "__main__":
    main()
