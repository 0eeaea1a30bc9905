#!/usr/bin/env python
"""bench.py -- RSPrompter inference hot path on B200 (contract: see the task brief / DESIGN.md section 6).

    python bench.py --gpus N --steps K --warmup W [--config NAME]   # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...         # the CPU oracle (reference arm)
    python bench.py ... --dump-outputs DIR                          # also write the last timed step's outputs as .npy

Configs (BASELINE.json `configs`):
    query_vith   (default) configs[2] / [3]: RSPrompter-query ViT-H bf16, bs 8 per GPU, 1024^2, 100 queries
    anchor_vitb            configs[1]:       RSPrompter-anchor ViT-B bf16, bs 8 per GPU, 1024^2
    anchor_vith, query_vitb                  the other two pairings
    maskrcnn_vitb          SAMSegMaskRCNN ViT-B (SAM encoder + RSFPN + stock Mask R-CNN heads), bs 8 per GPU, 1024^2
    mask2former_vitb       SAMSegMask2Former ViT-B (SAM encoder + RSFPN + stock Mask2Former head), bs 8 per GPU, 1024^2
    encoder_vith           configs[4]:       SAM ViT-H encoder only at --size {512,768,1024,1280}

A step is one full pass of one batch: uint8 images -> DetDataPreprocessor (fused into the patch-embed loader) -> SAM
ViT encoder -> RSFPN -> prompt head -> SAM mask decoder -> mask resize / threshold / score / box -> ONE result
record per rank (bit-packed masks + rows + counts) -> ONE all-gather of the records (issued on a side stream so it
overlaps the next step).  One process per GPU, batch-sharded (weak scaling).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

NUM_CLASSES, BATCH, SIZE, NQ = 10, 8, 1024, 100
N_INPUT_SETS = 6   # distinct uint8 input batches rotated through the timed loop (6 x 25 MB > 126 MB L2)
# DetDataPreprocessor of every rsprompter config (configs/rsprompter/_base_/rsprompter_anchor.py:39-48)
PREPROC = dict(type="DetDataPreprocessor", mean=[123.675, 116.28, 103.53], std=[58.395, 57.12, 57.375], bgr_to_rgb=True,
               pad_size_divisor=32)

CONFIGS = {
    "query_vith": dict(variant="query", arch="huge",
                       workload=f"RSPrompter-query ViT-H bf16, bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic, {NQ} queries "
                                f"(BASELINE.json configs[2]; configs[3] when batch-sharded over 8 GPUs)"),
    "anchor_vitb": dict(variant="anchor", arch="base",
                        workload=f"RSPrompter-anchor ViT-B bf16, bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic (BASELINE.json configs[1])"),
    "anchor_vith": dict(variant="anchor", arch="huge",
                        workload=f"RSPrompter-anchor ViT-H bf16, bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic"),
    "query_vitb": dict(variant="query", arch="base",
                       workload=f"RSPrompter-query ViT-B bf16, bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic, {NQ} queries"),
    "maskrcnn_vitb": dict(variant="maskrcnn", arch="base",
                          workload=f"SAM-seg Mask R-CNN ViT-B bf16 (SAMSegMaskRCNN), bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic"),
    "mask2former_vitb": dict(variant="mask2former", arch="base",
                             workload=f"SAM-seg Mask2Former ViT-B bf16 (SAMSegMask2Former), bs={BATCH}/GPU, {SIZE}x{SIZE} synthetic, {NQ} queries"),
    "encoder_vith": dict(variant="encoder", arch="huge",
                         workload="SAM-seg ViT-H encoder only (MMPretrainSamVisionEncoder), bs=%d/GPU, {S}x{S} synthetic "
                                  "(BASELINE.json configs[4])" % BATCH),
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return dict(tflops=float(p.get("bf16_tflops_sustained", p.get("bf16_tflops", 1400.0))),
                    hbm=float(p.get("hbm_gbs", 6650.0)), source="measured (MEASURED_PEAKS.json, sustained)")
    return dict(tflops=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md: 1.4 PF sustained, 6.65 TB/s)")


def _host_threads() -> int:
    """Threads this process may actually use: scheduler affinity, capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period))))
    except (OSError, ValueError):
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append(float(parts[0]))
                    self.max_mhz = float(parts[1])
                    for nm, v in zip(names, parts[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self):
        return dict(sm_mhz=statistics.median(self.samples) if self.samples else None, sm_max_mhz=self.max_mhz,
                    reasons=sorted(self.reasons), samples=len(self.samples))


def _workload_config(args, n_gpus: int) -> dict:
    c = CONFIGS[args.config]
    size = args.size if c["variant"] == "encoder" else SIZE
    cfg = dict(workload=c["workload"].replace("{S}", str(size)), config=args.config, image_size=size,
               num_classes=NUM_CLASSES, global_batch=BATCH * n_gpus,
               parallelism=f"dp{n_gpus} (batch-sharded, weights replicated)",
               l2_policy=f"{N_INPUT_SETS} distinct uint8 input batches rotated ({N_INPUT_SETS * BATCH * 3 * size * size >> 20} MB "
                         "in total; 126 MB L2); every step also streams tens of GB of activations through HBM, so "
                         "nothing of a step survives in L2 until the next",
               input="uint8 CHW images (PackDetInputs layout) through DetDataPreprocessor (BGR->RGB, mean/std)",
               weights="seeded random init of the exact architecture")
    return cfg


# ================================================================================================
# reference arm / CPU baseline: the oracle port on the host cores
# ================================================================================================
def _import_generators():
    """synthetic weight generators / arch tables WITHOUT executing the package __init__ (which maps librsp_b200.so):
    the reference arm must not load any of this repo's native code."""
    if "rsprompter_b200" in sys.modules:            # our own arm: the package is already imported
        from rsprompter_b200 import model_configs, sam_config, synthetic
        return synthetic, sam_config, model_configs
    import importlib
    import types
    pkg = types.ModuleType("rsprompter_b200")
    pkg.__path__ = [os.path.join(ROOT, "rsprompter_b200")]
    sys.modules["rsprompter_b200"] = pkg
    try:
        sam_config = importlib.import_module("rsprompter_b200.sam_config")
        synthetic = importlib.import_module("rsprompter_b200.synthetic")
        model_configs = importlib.import_module("rsprompter_b200.model_configs")
    finally:
        del sys.modules["rsprompter_b200"]           # leave no half-initialised package behind
    return synthetic, sam_config, model_configs


def _u8_images(n: int, size: int, seed: int) -> torch.Tensor:
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n, 3, size, size), generator=g, dtype=torch.uint8)


def _oracle_preprocess(u8: torch.Tensor) -> torch.Tensor:
    """DetDataPreprocessor arithmetic (data_preprocessor.py:110-148) in fp32 torch, for the CPU arm."""
    x = u8[:, [2, 1, 0]].float()
    mean = torch.tensor(PREPROC["mean"]).view(1, 3, 1, 1)
    std = torch.tensor(PREPROC["std"]).view(1, 3, 1, 1)
    return (x - mean) / std


def _oracle_setup(args):
    synthetic, sam_config, model_configs = _import_generators()
    c = CONFIGS[args.config]
    arch = sam_config.VISION_ARCHS[c["arch"]]
    sel = model_configs.SELECT_LAYERS[c["arch"]]
    darch = sam_config.SamDecoderArch()
    if c["variant"] == "anchor":
        from oracle import restate_anchor as ra
        sd = synthetic.anchor_detector_state_dict(arch, NUM_CLASSES, len(sel), seed=0)
        return lambda x: ra.anchor_predict(sd, arch, darch, x, NUM_CLASSES, sel)
    if c["variant"] == "maskrcnn":
        from oracle import restate_anchor as ra
        sd = synthetic.maskrcnn_detector_state_dict(arch, NUM_CLASSES, len(sel), seed=0)
        return lambda x: ra.maskrcnn_predict(sd, arch, x, NUM_CLASSES, sel)
    if c["variant"] == "mask2former":
        from oracle import restate_query as rq
        sd = synthetic.mask2former_detector_state_dict(arch, NUM_CLASSES, len(sel), nq=NQ, seed=0)
        return lambda x: rq.samseg_mask2former_predict(sd, arch, x, NUM_CLASSES, sel, max_per_image=NQ)
    if c["variant"] == "query":
        from oracle import restate_query as rq
        sd = synthetic.query_detector_state_dict(arch, NUM_CLASSES, len(sel), nq=NQ, seed=0)
        return lambda x: rq.query_predict(sd, arch, darch, x, NUM_CLASSES, sel, max_per_image=NQ)
    from dataclasses import replace
    from oracle import restate
    arch = sam_config.vision_arch(c["arch"], img_size=args.size)
    sd = synthetic.vision_encoder_state_dict(arch, seed=0)
    return lambda x: restate.vit_encoder(sd, replace(arch, output_hidden_states=False), x)


def cpu_baseline(args, max_seconds: float = 60.0) -> dict:
    """Oracle ('port') on the host cores, bounded sample: the whole pipeline on 1 image (bs=1) of the workload."""
    cores = _host_threads()
    torch.set_num_threads(cores)
    run = _oracle_setup(args)
    size = args.size if CONFIGS[args.config]["variant"] == "encoder" else SIZE
    x = _oracle_preprocess(_u8_images(1, size, 0))
    with torch.no_grad():
        t0 = time.perf_counter()
        run(x)
        dt = time.perf_counter() - t0
        if dt < max_seconds / 3:   # one more for a steadier number if cheap
            t0 = time.perf_counter()
            run(x)
            dt = time.perf_counter() - t0
    return dict(value=1.0 / dt, unit="images/s", cores=cores, kind="port",
                sample=f"full {args.config} pipeline (oracle/restate*.py, fp32, torch {torch.__version__}, {cores} threads) "
                       f"on 1 image {size}x{size}, bs=1, {dt:.1f} s")


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _host_threads()
    torch.set_num_threads(cores)
    run = _oracle_setup(args)
    size = args.size if CONFIGS[args.config]["variant"] == "encoder" else SIZE
    xs = [_oracle_preprocess(_u8_images(1, size, s)) for s in range(2)]
    budget = 60.0      # seconds of warmup at most
    t_start = time.perf_counter()
    w_done = 0
    times = []
    with torch.no_grad():
        for i in range(args.warmup):
            run(xs[i % 2])
            w_done += 1
            if time.perf_counter() - t_start > budget:
                break
        for i in range(args.steps):
            t0 = time.perf_counter()
            run(xs[i % 2])
            times.append(time.perf_counter() - t0)
    total = sum(times)
    val = len(times) / total
    line = dict(metric="images/sec", value=val, unit="images/s", n_gpus=args.gpus, steps=len(times),
                warmup=w_done, ms_per_step=1e3 * total / len(times), higher_is_better=True, scaling="weak",
                vs_baseline=None, dtype="f32", data="synthetic", impl="reference",
                config=_workload_config(args, args.gpus),
                cpu_baseline=dict(value=val, unit="images/s", cores=cores, kind="port",
                                  sample=f"each step = full {args.config} pipeline on 1 image (bs=1) of the workload, "
                                         f"{cores} host threads (affinity / cgroup quota); {len(times)} timed steps, "
                                         f"step times {min(times):.2f}-{max(times):.2f} s"),
                e2e=dict(value=val, unit="images/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                native_so_loaded=any("librsp_b200" in ln for ln in open("/proc/self/maps")))
    print(json.dumps(line))


# ================================================================================================
# this repo's arm
# ================================================================================================
KERNEL_GROUPS = (("gemm", "gemm_bf16_tcgen05"), ("attention_global", "vit_attention_kernel"),
                 ("attention_window", "vit_window_attention_kernel"))


def _profile_kernels(step_fn, n_steps: int) -> list:
    """Per-kernel device durations of n_steps steps from CUPTI activity records (torch.profiler): works for kernels
    replayed from a CUDA graph, costs nothing inside the kernels, and is not used for any timed number."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(n_steps):
            step_fn(i)
        torch.cuda.synchronize()
    fd, path = tempfile.mkstemp(suffix=".json")
    os.close(fd)
    try:
        prof.export_chrome_trace(path)
        with open(path) as f:
            tr = json.load(f)
    finally:
        os.unlink(path)
    ev = [e for e in tr.get("traceEvents", []) if e.get("cat") in ("kernel", "Kernel") and "dur" in e]
    ev.sort(key=lambda e: e["ts"])
    return [(e["name"], float(e["dur"]) * 1e-3) for e in ev]     # (name, ms)


def _roofline(model_step, trace_fn, inst_steps: int, step_ms: float, peaks: dict, args) -> dict:
    """roofline of the dominant kernel family (the tcgen05 GEMM): sum(2MNK) / sum(kernel time), plus the encoder-only
    GEMM figure, the attention kernels and the whole step (SURVEY 8(d) i-iii)."""
    from rsprompter_b200 import _lib
    _lib.trace = []
    trace_fn()
    torch.cuda.synchronize()
    trace, _lib.trace = _lib.trace, None
    kernels = _profile_kernels(model_step, inst_steps)
    total_ms = sum(t for _, t in kernels) / inst_steps
    out = dict(bound="tensor", kernel="gemm_bf16_tcgen05_*_kernel (all tile shapes / epilogues)", peak=peaks["tflops"],
               unit="TFLOP/s", peak_source=peaks["source"],
               method="per-kernel durations from CUPTI activity records of %d graph-replayed steps; FLOP = 2*M*N*K "
                      "(4*T^2*hd per head for attention) logged per launch" % inst_steps,
               kernel_ms_per_step=total_ms, kernels_per_step=len(kernels) // inst_steps)
    groups = {}
    for gname, pat in KERNEL_GROUPS:
        ts = [t for n, t in kernels if pat in n]
        want = [r for r in trace if r["kind"] == gname]
        g = dict(launches_per_step=len(ts) // inst_steps, ms_per_step=sum(ts) / inst_steps,
                 tflop_per_step=sum(r["flops"] for r in want) / 1e12)
        g["tflops"] = g["tflop_per_step"] / (g["ms_per_step"] * 1e-3) if g["ms_per_step"] > 0 else 0.0
        g["frac"] = g["tflops"] / peaks["tflops"]
        g["launch_count_matches_trace"] = len(ts) == len(want) * inst_steps
        if gname == "gemm" and g["launch_count_matches_trace"]:      # per-scope split through launch order
            n = len(want)
            for scope in sorted({r["scope"] for r in want}):
                idx = [i for i, r in enumerate(want) if r["scope"] == scope]
                ms = sum(ts[s * n + i] for s in range(inst_steps) for i in idx) / inst_steps
                fl = sum(want[i]["flops"] for i in idx) / 1e12
                groups[f"gemm[{scope}]"] = dict(launches_per_step=len(idx), ms_per_step=ms, tflop_per_step=fl,
                                                tflops=fl / (ms * 1e-3) if ms > 0 else 0.0,
                                                frac=fl / (ms * 1e-3) / peaks["tflops"] if ms > 0 else 0.0)
        groups[gname] = g
    import collections
    import re
    agg = collections.defaultdict(lambda: [0, 0.0])
    for n, t in kernels:
        short = re.sub(r"^void |rsp::|v2::|win::", "", n)
        short = re.sub(r"\(.*", "", short)[:70]
        agg[short][0] += 1
        agg[short][1] += t
    out["top_kernels"] = [dict(kernel=k, launches_per_step=v[0] / inst_steps, ms_per_step=v[1] / inst_steps)
                          for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])[:14]]
    gm = groups["gemm"]
    out.update(achieved=gm["tflops"], frac=gm["frac"], launches_per_step=gm["launches_per_step"],
               gemm_ms_per_step=gm["ms_per_step"], algorithmic_tflop_per_step=gm["tflop_per_step"], groups=groups)
    tfl = sum(r["flops"] for r in trace) / 1e12
    out["whole_step"] = dict(tflop_per_step=tfl, ms_per_step=step_ms, tflops=tfl / (step_ms * 1e-3),
                             frac=tfl / (step_ms * 1e-3) / peaks["tflops"])
    # a dominant-kernel time above the step time would mean the measurement is broken (round-1 bug): refuse it
    assert gm["ms_per_step"] <= step_ms * 1.02, f"GEMM time {gm['ms_per_step']:.2f} ms exceeds the step {step_ms:.2f} ms"
    # ncu dram bytes of the same step, per GEMM launch, from the committed capture (null until one exists)
    out["traffic"], out["traffic_source"] = None, None
    tpath = os.path.join(ROOT, "profiles", f"r02_traffic_{args.config}.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        g = [k for k in tj["kernels"] if "gemm_bf16_tcgen05" in k["kernel"]]
        if g:
            out["traffic"] = sum(k["dram_read_bytes"] + k["dram_write_bytes"] for k in g) / sum(k["launches"] for k in g)
            out["traffic_source"] = f"profiles/r02_traffic_{args.config}.json (ncu capture of one step, mean bytes per GEMM launch)"
    return out


DUMP_BYTES = 64 << 20      # --dump-outputs writes at most this much
MASK_SAMPLE = 4096         # mask pixels per instance slot written by --dump-outputs (the same seeded positions for all)


def dump_outputs(out_dir: str, host_buf: torch.Tensor, rec0, variant: str, size: int) -> None:
    """Write what one end-to-end step handed its caller in host memory (rank 0's batch) as DIR/<name>.npy.

    encoder:   image_embeddings  f32 [B, 256, S/16, S/16] (a flat seeded sample if larger than DUMP_BYTES)
    detectors: counts f64 [B]; rows f32 [B, M, 6] (x1, y1, x2, y2, score, label); mask_area f64 [B, M] (set pixels of
               each mask); mask_sample f32 [B, M, MASK_SAMPLE] (each mask at MASK_SAMPLE pixels drawn with seed 0).
               Slots at or beyond an image's count are written as zeros."""
    import numpy as np
    g = torch.Generator().manual_seed(0)
    if variant == "encoder":
        emb = host_buf.view(torch.float32).view(BATCH, 256, size // 16, size // 16)
        if emb.numel() * 4 > DUMP_BYTES:
            idx = torch.randperm(emb.numel(), generator=g)[:DUMP_BYTES // 4].sort().values
            arrays = dict(image_embeddings_sample=emb.reshape(-1)[idx])
        else:
            arrays = dict(image_embeddings=emb)
    else:
        rec = rec0.like(host_buf)
        H, W = rec.hw
        valid = torch.arange(rec.slots)[None, :] < rec.counts[:, None].long()
        bits = rec.mask_bits.reshape(rec.batch, rec.slots, H * W // 8)
        pix = torch.randperm(H * W, generator=g)[:MASK_SAMPLE]
        sample = (bits[..., pix // 8] >> (pix % 8).to(torch.uint8)) & 1
        area = sum(((bits >> k) & 1).sum(-1, dtype=torch.int64) for k in range(8))
        v = valid[..., None]
        arrays = dict(counts=rec.counts.double(), rows=torch.where(v, rec.rows, 0.0),
                      mask_area=torch.where(valid, area.double(), 0.0), mask_sample=torch.where(v, sample.float(), 0.0))
    assert sum(a.numel() * a.element_size() for a in arrays.values()) <= DUMP_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a.contiguous().numpy())


def run_ours(args) -> None:
    import torch.distributed as dist
    from rsprompter_b200 import _lib, model_configs, sam_config, synthetic
    from rsprompter_b200.model_configs import SELECT_LAYERS
    from rsprompter_b200.registry import MODELS
    from rsprompter_b200.results import ResultRecord

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (the CUDA path has no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    c = CONFIGS[args.config]
    variant, arch_name = c["variant"], c["arch"]
    size = args.size if variant == "encoder" else SIZE
    use_graph = not os.environ.get("RSP_BENCH_NO_GRAPH")
    n_sel = len(SELECT_LAYERS[arch_name])
    if variant == "encoder":
        model = MODELS.build(dict(type="MMPretrainSamVisionEncoder", hf_pretrain_name=f"facebook/sam-vit-{arch_name}",
                                  img_size=size))
        arch = model.vision_encoder.arch
        model.vision_encoder.load_state_dict(synthetic.vision_encoder_state_dict(arch, seed=0))
        model = model.to(dev)
        prep = MODELS.build(dict(PREPROC)).to(dev)
    else:
        arch = sam_config.VISION_ARCHS[arch_name]
        if variant == "anchor":
            cfg = model_configs.anchor_model_cfg(arch_name, NUM_CLASSES)
            sd = synthetic.anchor_detector_state_dict(arch, NUM_CLASSES, n_sel, seed=0)
        elif variant == "maskrcnn":
            cfg = model_configs.maskrcnn_model_cfg(arch_name, NUM_CLASSES)
            sd = synthetic.maskrcnn_detector_state_dict(arch, NUM_CLASSES, n_sel, seed=0)
        elif variant == "mask2former":
            cfg = model_configs.mask2former_model_cfg(arch_name, NUM_CLASSES, num_queries=NQ)
            sd = synthetic.mask2former_detector_state_dict(arch, NUM_CLASSES, n_sel, nq=NQ, seed=0)
        else:
            cfg = model_configs.query_model_cfg(arch_name, NUM_CLASSES, prompt_shape=(NQ, 5))
            sd = synthetic.query_detector_state_dict(arch, NUM_CLASSES, n_sel, nq=NQ, seed=0)
        cfg["data_preprocessor"] = dict(PREPROC)
        model = MODELS.build(cfg)
        model.load_state_dict(sd)
        model = model.to(dev)
        prep = model.data_preprocessor
        if use_graph:
            model.enable_cuda_graphs()      # the device-resident forward is captured once per input shape and replayed

    host = [_u8_images(BATCH, size, 1000 + 10 * rank + s).pin_memory() for s in range(N_INPUT_SETS)]
    # resident arm: what the data preprocessor hands the detector (the uint8 batch with the normalisation attached)
    resident = [prep(dict(inputs=h.to(dev)), False, fuse_patch_embed=True)["inputs"] for h in host]
    side = torch.cuda.Stream()
    M = NQ if variant in ("query", "mask2former") else 100

    enc_graphs = {}

    def encoder_forward(x):
        """encoder-only config: CUDA-graph replay of MMPretrainSamVisionEncoder.forward (static shapes, no host sync)."""
        if not use_graph:
            return model(x)[0]
        if "g" not in enc_graphs:
            static_in = x.clone()
            static_in.rsp_norm = x.rsp_norm
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                for _ in range(2):
                    model(static_in)
            torch.cuda.current_stream().wait_stream(s)
            g = torch.cuda.CUDAGraph()
            n0 = _lib.launch_count
            with torch.cuda.graph(g):
                out = model(static_in)[0]
            enc_graphs.update(g=g, inp=static_in, out=out, n=_lib.launch_count - n0)
        enc_graphs["inp"].copy_(x, non_blocking=True)
        enc_graphs["g"].replay()
        _lib.launch_count += enc_graphs["n"]
        return enc_graphs["out"]

    # ---- the step: forward + post-process into a record, then the record leaves on the side stream ------------
    if variant == "encoder":
        emb_bytes = BATCH * 256 * (size // 16) ** 2 * 4
        gbuf = [torch.empty(world, emb_bytes, dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
        hbuf = [torch.empty(emb_bytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        d2h_bytes = emb_bytes
    else:
        rec0 = ResultRecord(BATCH, M, (size, size), device=dev)
        gbuf = [torch.empty(world, rec0.nbytes, dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
        hbuf = [torch.empty(rec0.nbytes, dtype=torch.uint8).pin_memory() for _ in range(2)]
        d2h_bytes = rec0.nbytes
    side_done = [None, None]

    def compute(x):
        if variant == "encoder":
            return encoder_forward(x)
        return model.predict_records(x)

    def leave(i, result, to_host: bool):
        """gather (and, end to end, the D2H copy) of step i's result on the side stream; buffers alternate."""
        if world == 1 and not to_host:
            return
        ev = torch.cuda.Event()
        ev.record()
        side.wait_event(ev)
        with torch.cuda.stream(side):
            buf = result.buf if variant != "encoder" else result.view(-1).view(torch.uint8)
            if world > 1:
                dist.all_gather_into_tensor(gbuf[i % 2].view(-1), buf)
            if to_host:
                hbuf[i % 2].copy_(buf, non_blocking=True)
            done = torch.cuda.Event()
            done.record()
        side_done[i % 2] = done

    def step_resident(i):
        if side_done[i % 2] is not None:        # the buffer pair written two steps ago must have left
            torch.cuda.current_stream().wait_event(side_done[i % 2])
        leave(i, compute(resident[i % N_INPUT_SETS]), to_host=False)

    def step_e2e(i):
        if side_done[i % 2] is not None:
            torch.cuda.current_stream().wait_event(side_done[i % 2])
        if variant == "encoder":
            x = prep(dict(inputs=host[i % N_INPUT_SETS]), False, fuse_patch_embed=True)["inputs"]
            leave(i, encoder_forward(x), to_host=True)
        else:   # the user-facing call: uint8 host batch -> data preprocessor -> predict -> record -> host
            data = model._preprocess(dict(inputs=host[i % N_INPUT_SETS]))
            leave(i, model.predict_records(data["inputs"]), to_host=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        torch.cuda.current_stream().wait_stream(side)      # every gather / D2H is inside the timed region
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    warm = max(args.warmup, 3)
    for i in range(warm):
        step_resident(i)
    for i in range(2):
        step_e2e(i)
    barrier()

    with ClockSampler(local) as clk:
        l0 = _lib.launch_count
        ms = timed(step_resident, args.steps)
        launches = _lib.launch_count - l0
        ms_e2e = timed(step_e2e, args.steps)
    if args.dump_outputs and rank == 0:     # the host buffer the last timed step's record / embedding was copied to
        dump_outputs(args.dump_outputs, hbuf[(args.steps - 1) % 2], None if variant == "encoder" else rec0,
                     variant, size)

    peaks = _peaks()
    roof, roof_err = None, None
    if rank == 0 and not os.environ.get("RSP_BENCH_SKIP_ROOFLINE"):
        enc = model.vision_encoder if variant == "encoder" else model.backbone.vision_encoder
        orig_encode = enc.encode

        def scoped_encode(*a, **k):
            _lib.trace_scope = "encoder"
            try:
                return orig_encode(*a, **k)
            finally:
                _lib.trace_scope = "heads"

        def trace_fn():      # one eager forward with the launch log on: (kind, scope, flops) per tensor-core launch
            enc.encode = scoped_encode
            _lib.trace_scope = "heads"
            try:
                if variant == "encoder":
                    model(resident[0])
                else:
                    model.predict_raw(resident[0])
            finally:
                enc.encode = orig_encode
        try:
            roof = _roofline(lambda i: compute(resident[i % N_INPUT_SETS]), trace_fn, min(args.steps, 3),
                             ms / args.steps, peaks, args)
        except Exception as e:  # noqa: BLE001  (CUPTI unavailable etc.: report, do not fake)
            roof_err = f"{type(e).__name__}: {e}"
    if world > 1:
        dist.barrier()

    if rank == 0:
        imgs = BATCH * world * args.steps
        value = imgs / (ms * 1e-3)
        e2e_val = imgs / (ms_e2e * 1e-3)
        h2d = BATCH * 3 * size * size
        cb = cpu_baseline(args) if (world == 1 and not os.environ.get("RSP_BENCH_SKIP_CPU")) else None
        line = dict(metric="images/sec", value=value, unit="images/s", n_gpus=world, steps=args.steps,
                    warmup=warm, ms_per_step=ms / args.steps, higher_is_better=True,
                    scaling="weak", vs_baseline=None, dtype="bf16", data="synthetic",
                    config=_workload_config(args, world), clocks=clk.summary(), cuda_graph=use_graph,
                    e2e=dict(value=e2e_val, unit="images/s", h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h_bytes,
                             ms_per_step=ms_e2e / args.steps,
                             note="pinned uint8 host batch -> DetDataPreprocessor (fused) -> predict -> result record "
                                  "(bit-packed 1024^2 masks + rows + counts) -> pinned host buffer, every step; the "
                                  "record copy / all-gather run on a side stream and are complete inside the timed region"),
                    collective=(f"1 all_gather_into_tensor per step of the {d2h_bytes} B per-rank result record"
                                if world > 1 else None),
                    gpu_launches=launches, roofline=roof)
        if roof_err:
            line["roofline_error"] = roof_err
        if cb is not None:
            line["cpu_baseline"] = cb
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="query_vith", choices=sorted(CONFIGS))
    ap.add_argument("--size", type=int, default=1024, help="image size of the encoder_vith config (512/768/1024/1280)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last end-to-end step returned (rank 0's batch) as "
                         "DIR/<name>.npy, float32 / float64, at most 64 MB; the inputs are seeded, so runs with the "
                         "same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
