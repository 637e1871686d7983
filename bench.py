#!/usr/bin/env python
"""bench.py — PLIP dual-tower inference throughput on B200 (BASELINE.json metric: image-text pairs/s).

    python bench.py --gpus N --steps K --warmup W                      # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K --warmup W     # the reference's own CPU path
    python bench.py --config cfg3|cfg4|cfg5 ...                        # BASELINE.json configs[2..4] as their own lines
    python bench.py ... --dump-outputs DIR                             # also write the last timed step's outputs (.npy)

Default workload ("pairs"): one step per GPU = one pass of the hot path over 1024 synthetic image-text pairs:
vision tower (224x224, bf16 pixels resident in HBM) + text tower (77-token ids) + L2-normalise + logits_per_image
against the captions of ALL ranks (NCCL all-gather of the text embeddings when N > 1) — through
``ShardedCLIP.clip_forward``.  ``value`` = pairs/s with inputs resident in HBM; ``e2e`` = the same step through the
product API (``PlipCLIPModel.__call__`` / ``ShardedCLIP.clip_forward``) on pinned HOST inputs (uint8 tiles + int64
ids): H2D of every step's inputs and the D2H of its logits are inside the timed region.  ``roofline`` reports the
dominant kernel timed INSIDE the step (CUDA event pairs on the launch stream, ``plip_profile_*``).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PAIRS = 1024                      # images / captions per step per GPU (BASELINE cfg2/cfg3 micro-batch)
FLOP_IMG = 8.81762e9              # SURVEY.md §8: dense FLOPs per image (vision tower + projection)
FLOP_TXT = 5.95954e9              # per 77-token caption
METRIC = "image-text pairs/sec (224x224, 77-tok)"

WORKLOADS = {
    "pairs": "dual tower + logits_per_image: 1024 images (224x224, bf16 NCHW) x 1024 captions (77 tokens) per step per GPU, "
             "ViT-B/32 PLIP geometry, seeded random weights (plip_b200.synthetic.make_state_dict(0))",
    "cfg3": "BASELINE configs[2]: dual tower + logits_per_image, 4096 images x 1024 captions (77 tokens) per step, 1 GPU",
    "cfg4": "BASELINE configs[3]: zero-shot classification, 100000 synthetic uint8 tiles x 64 class prompts, images "
            "batch-sharded over the GPUs, all-gather of the image embeddings",
    "cfg5": "BASELINE configs[4]: image->text retrieval, 1000000-tile gallery + 10000 text queries, gallery and queries "
            "sharded over the GPUs, all-gather of the query embeddings, full similarity matrix row-sharded",
}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return {"bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "hbm_gbs": p["hbm_gbs"], "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        # samples inside the timed region; a region shorter than the 100 ms sampling period falls back to the samples
        # taken right around it (the GPU is under the same load during the warm-up just before)
        rows = ([r for t, r in self.rows if t0 - 0.05 <= t <= t1 + 0.05] or
                [r for t, r in self.rows if t0 - 0.35 <= t <= t1 + 0.25] or [r for _, r in self.rows][-3:])
        sm, mx, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def usable_cores() -> int:
    """Host cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per) + 0.5)))
    except Exception:  # noqa: BLE001
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, int(q / per + 0.5)))
        except Exception:  # noqa: BLE001
            pass
    return max(1, min(n, int(os.environ.get("PLIP_BENCH_MAX_THREADS", "256"))))


def _dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def config_dict(name: str, ws: int):
    cfg = {"workload": WORKLOADS[name], "name": name, "seq_len": 77, "parallelism": f"dp{ws}"}
    if name == "pairs":
        cfg.update({"pairs_per_step_per_gpu": PAIRS,
                    "l2_policy": "inputs alternate between 2 resident sets; pixels 308 MB/step > 126 MB L2",
                    "collective": "all_gather of text embeddings [1024,512] f32 per rank (NCCL)" if ws > 1 else "none"})
    elif name == "cfg3":
        cfg.update({"images_per_step": 4096, "captions_per_step": 1024,
                    "l2_policy": "4 distinct micro-batches of 1024 images (1.2 GB of pixels) per step > 126 MB L2"})
    elif name == "cfg4":
        cfg.update({"tiles": 100000, "prompts": 64, "l2_policy": "every tile distinct (15 GB of uint8 tiles in HBM)",
                    "collective": "all_gather of image embeddings [12500,512] f32 per rank (NCCL)" if ws > 1 else "none"})
    elif name == "cfg5":
        cfg.update({"gallery": 1000000, "queries": 10000,
                    "l2_policy": "gallery tiles drawn cyclically from a resident pool of 8192 distinct uint8 tiles per rank "
                                 "(1.2 GB >> 126 MB L2; 150 GB of distinct tiles would not fit beside the 40 GB result at N=1)",
                    "collective": "all_gather of query embeddings [10000/N,512] f32 per rank (NCCL)" if ws > 1 else "none"})
    return cfg


# =================================================================================================
# reference arm: the reference's own CPU path (live transformers.CLIPModel behind the restated PLIP loop)
# =================================================================================================
class CpuReference:
    """fp32 CLIPModel on the host cores.  kind = "reference" when the live ``transformers`` package (the code the
    reference delegates its arithmetic to, plip.py:7,26) runs it, "port" when only ``oracle/clip_oracle.py`` can."""

    def __init__(self, sd):
        from oracle import ref_cpu
        self.sd, self.ref_cpu = sd, ref_cpu
        try:
            import transformers
            self.model = ref_cpu.load_model(sd)
            self.kind = "reference"
            self.how = (f"live transformers {transformers.__version__} CLIPModel fp32 (the package plip.py:26,50,68 delegates to), "
                        "driven by oracle/ref_cpu.py (restated plip.py batch loop / README model(**inputs) call)")
        except Exception as exc:  # noqa: BLE001
            self.model = None
            self.kind = "port"
            self.how = f"oracle/clip_oracle.py (torch-CPU restatement of CLIPModel.forward); transformers unavailable: {exc}"[:300]

    def forward(self, ids, px, mask=None):
        if self.model is not None:
            return self.ref_cpu.clip_forward(self.model, ids, px, mask)
        from oracle import clip_oracle as O
        return O.clip_forward(self.sd, ids, px, mask)["logits_per_image"]

    def images(self, px, bs):
        if self.model is not None:
            return self.ref_cpu.plip_encode_images(self.model, px, bs)
        from oracle import clip_oracle as O
        return torch.cat([O.get_image_features(self.sd, px[i:i + bs]) for i in range(0, px.shape[0], bs)]).numpy()

    def text(self, ids, mask, bs):
        if self.model is not None:
            return self.ref_cpu.plip_encode_text(self.model, ids, mask, bs)
        from oracle import clip_oracle as O
        return torch.cat([O.get_text_features(self.sd, ids[i:i + bs], mask[i:i + bs] if mask is not None else None)
                          for i in range(0, ids.shape[0], bs)]).numpy()


def reference_sample(name: str, ref: CpuReference, synth):
    """A bounded sample of the named workload for the CPU legs: returns (callable, units per call, description).
    Batch 32 on the host cores, BASELINE.md §3."""
    bs = 32
    px = synth.pixel_values(bs)
    if name == "pairs":
        ids, mask = synth.token_ids(bs, full_length=True)
        return (lambda: ref.forward(ids, px, mask)), bs, f"{bs} images x {bs} captions per step: model(**inputs).logits_per_image"
    if name == "cfg3":
        ids, mask = synth.token_ids(bs // 4)
        return (lambda: ref.forward(ids, px, mask)), bs, f"{bs} images x {bs // 4} captions per step (cfg3's 4:1 ratio): model(**inputs)"
    if name == "cfg4":
        ids, mask = synth.token_ids(64, seed=1235)

        def zs():
            t = ref.text(ids, mask, 8)                                 # plip.py:95: encode_text(labels, batch_size=8)
            i = ref.images(px, 8)                                      # plip.py:97
            i = i / np.linalg.norm(i, axis=-1, keepdims=True)          # plip.py:73-76
            return np.argmax(i @ t.T, axis=-1)                         # plip.py:102
        return zs, bs, f"{bs} tiles x 64 prompts per step: PLIP.zero_shot_classification flow (plip.py:89-103), batch_size 8"
    if name == "cfg5":
        ids, mask = synth.token_ids(8, seed=1235)

        def rt():
            g = ref.images(px, 32)
            q = ref.text(ids, mask, 8)
            q = q / np.linalg.norm(q, axis=-1, keepdims=True)
            return (q @ g.T).argsort()[:, -10:][:, ::-1]               # plip.py:85
        return rt, bs, f"{bs} gallery tiles + 8 queries per step: encode_images + encode_text + _nearest_neighbours (plip.py:78-87)"
    raise ValueError(name)


def setup_cpu_reference(name: str):
    from oracle import synth, weights
    torch.set_grad_enabled(False)
    cores = usable_cores()
    sd = weights.make_state_dict(0)
    ref = CpuReference(sd)
    fn, units, what = reference_sample(name, ref, synth)
    from oracle import ref_cpu
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores} | {cores})
    best, times = ref_cpu.pick_threads(fn, cands)
    return sd, ref, fn, units, what, best, times, cores


def run_reference(args):
    rank, _, ws = _dist_env()
    if rank != 0:
        return 0
    sd, ref, fn, units, what, threads, sweep, cores = setup_cpu_reference(args.config)
    for _ in range(max(1, min(args.warmup, 2))):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = time.perf_counter() - t0
    val = units * args.steps / dt
    metric, unit = metric_of(args.config)
    line = {"impl": "reference", "metric": metric, "value": val, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak" if args.config == "pairs" else "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_dict(args.config, max(1, args.gpus)),
            "cpu_baseline": {"value": val, "unit": unit, "cores": threads, "kind": ref.kind,
                             "sample": f"{args.steps} steps, each a bounded sample of the workload: {what}; {ref.how}; "
                                       f"{threads} threads (fastest of a one-shot sweep {{threads: s}} = "
                                       f"{ {k: round(v, 3) for k, v in sweep.items()} } on {cores} usable cores)"},
            "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


def metric_of(name: str):
    if name in ("pairs", "cfg3"):
        return METRIC, "pairs/s"
    if name == "cfg4":
        return "zero-shot classified tiles/sec (224x224 tiles x 64 prompts)", "images/s"
    return "retrieval gallery tiles/sec (1M gallery x 10k queries, full similarity matrix)", "images/s"


# =================================================================================================
# this repo's arm
# =================================================================================================
def cpu_baseline_sample(name: str):
    sd, ref, fn, units, what, threads, sweep, cores = setup_cpu_reference(name)
    _, unit = metric_of(name)
    t0 = time.perf_counter()
    reps = 0
    while reps < 2 or (time.perf_counter() - t0 < 12.0 and reps < 24):
        fn()
        reps += 1
    dt = time.perf_counter() - t0
    return sd, {"value": units * reps / dt, "unit": unit, "cores": threads, "kind": ref.kind,
                "sample": f"{reps} x ({what}); fp32, torch {torch.__version__} CPU; {ref.how}; {threads} threads (fastest of "
                          f"{ {k: round(v, 3) for k, v in sweep.items()} } s on {cores} usable cores)"}


def kernel_bursts(eng, peaks, stream):
    """The four layer GEMM shapes of the vision tower, each timed ALONE in short bursts (-> burst peak)."""
    from plip_b200._lib import check
    L = eng._L
    M = PAIRS * 50
    shapes = [("ln1+qkv", 5, 2304, 768), ("out_proj+resid", 2, 768, 768), ("ln2+fc1+gelu", 6, 3072, 768),
              ("fc2+resid", 2, 768, 3072)]
    res = []
    stats = torch.zeros(M, 8, 2, device="cuda")
    stats[:, 0, 1] = 768.0                                   # mean 0, var 1 -> rstd ~ 1
    for name, epi, N, K in shapes:
        A = torch.randn(M, K, device="cuda").to(torch.bfloat16)
        W = (torch.randn(N, K, device="cuda") * 0.03).to(torch.bfloat16)
        bias = torch.zeros(N, device="cuda")
        colsum = W.float().sum(1).contiguous()
        out = torch.zeros(M, N, device="cuda", dtype=torch.float32 if epi == 2 else torch.bfloat16)
        xb = torch.empty(M, N, device="cuda", dtype=torch.bfloat16) if epi == 2 else None
        st_out = torch.empty(M, 8, 2, device="cuda") if epi == 2 else None
        call = lambda: check(L.plip_dbg_gemm(A.data_ptr(), K, W.data_ptr(), K, M, N, K, bias.data_ptr(), out.data_ptr(), N,  # noqa: E731
                                             None, epi, 0, 0, colsum.data_ptr() if epi >= 5 else None,
                                             stats.data_ptr() if epi >= 5 else None, 1 if epi >= 5 else 0,
                                             xb.data_ptr() if xb is not None else None,
                                             st_out.data_ptr() if st_out is not None else None, stream), "gemm")
        for _ in range(3):
            call()
        bursts = []
        for _ in range(6):          # MEASURED_PEAKS' burst protocol: best of short bursts separated by pauses
            time.sleep(0.03)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                call()
            e1.record()
            torch.cuda.synchronize()
            bursts.append(e0.elapsed_time(e1) / 3)
        ms = min(bursts)
        tf = 2.0 * M * N * K / ms / 1e9
        hbm = (M * K * 2 + N * K * 2 + (M * N * 10 if epi == 2 else M * N * 2)) / ms / 1e6
        res.append({"kernel": f"gemm_tcgen05[{name}]", "M": M, "N": N, "K": K, "us": ms * 1e3, "tflops": tf,
                    "frac_of_burst_peak": tf / peaks["bf16_tflops"], "GBps": hbm, "frac_of_hbm_peak": hbm / peaks["hbm_gbs"],
                    "us_mean": sum(bursts) / len(bursts) * 1e3})
        del A, W, out, xb, st_out
    return res


def in_step_profile(eng, run_step, peaks, reps=3):
    """Average duration of every kernel role INSIDE the step (event pairs on the launch stream), with its roofline."""
    for _ in range(2):
        run_step()
    torch.cuda.synchronize()
    eng.profile(True)
    for _ in range(reps):
        run_step()
    torch.cuda.synchronize()
    rows = eng.profile_read()
    eng.profile(False)
    tot = sum(r["total_ms"] for r in rows) or 1.0
    out = []
    for r in rows:
        n = max(1, r["launches"])
        us = r["total_ms"] / n * 1e3
        t_tensor = r["flops"] / n / (peaks["bf16_tflops_sustained"] * 1e12) * 1e6      # us at the sustained tensor peak
        t_hbm = r["bytes"] / n / (peaks["hbm_gbs"] * 1e9) * 1e6                          # us at the measured HBM peak
        bound = "tensor" if t_tensor >= t_hbm else "hbm"
        out.append({"kernel": r["name"], "launches_per_step": r["launches"] / reps, "us": us, "share_of_step": r["total_ms"] / tot,
                    "tflops": r["flops"] / n / us / 1e6 if r["flops"] else 0.0, "GBps": r["bytes"] / n / us / 1e3,
                    "bound": bound, "frac_of_roofline": max(t_tensor, t_hbm) / us if us > 0 else None,
                    "algorithmic_flops_per_launch": r["flops"] / n, "algorithmic_bytes_per_launch": r["bytes"] / n})
    return out


def roofline_from_profile(prof, peaks, traffic_json):
    """`roofline` = the kernel role with the largest share of the step; `roofline_worst` = the layer kernel furthest
    below its own roofline.  Both timed inside the step -> sustained tensor peak / measured HBM peak."""
    layer = [p for p in prof if p["share_of_step"] > 0.02]
    if not layer:
        return None, None
    dom = max(layer, key=lambda p: p["share_of_step"])
    worst = min(layer, key=lambda p: p["frac_of_roofline"] or 1.0)

    def obj(p):
        tr = None
        if traffic_json:
            key = p["kernel"].split("/", 1)[1]
            tower = p["kernel"].split("/", 1)[0]
            ent = traffic_json.get(f"{tower}/{key}") or traffic_json.get(key)
            if isinstance(ent, dict) and "traffic_mb" in ent:
                tr = ent["traffic_mb"] * 1e6
        if p["bound"] == "tensor":
            return {"bound": "tensor", "achieved": p["tflops"], "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                    "frac": p["tflops"] / peaks["bf16_tflops_sustained"], "traffic": tr, "kernel": p["kernel"],
                    "us_per_launch_in_step": p["us"], "share_of_step": p["share_of_step"],
                    "frac_of_burst_peak": p["tflops"] / peaks["bf16_tflops"],
                    "algorithmic_flops_per_launch": p["algorithmic_flops_per_launch"],
                    "peak_source": peaks["source"] + ", sustained figure (kernel timed inside the step with CUDA event pairs "
                                                     "on the launch stream)"}
        return {"bound": "hbm", "achieved": p["GBps"], "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": p["GBps"] / peaks["hbm_gbs"], "traffic": tr, "kernel": p["kernel"], "us_per_launch_in_step": p["us"],
                "share_of_step": p["share_of_step"], "algorithmic_bytes_per_launch": p["algorithmic_bytes_per_launch"],
                "peak_source": peaks["source"] + " (kernel timed inside the step with CUDA event pairs on the launch stream)"}
    return obj(dom), obj(worst)


def stock_pytorch_context(sd, dev):
    """Context line (SURVEY.md §8d): transformers.CLIPModel moved to the same GPU in bfloat16 (stock cuBLAS / SDPA kernels)
    on the same 1024-pair step.  Not on any product path; skipped silently if transformers is unavailable."""
    try:
        from transformers import CLIPConfig, CLIPModel
        from plip_b200 import synthetic as synth
        m = CLIPModel(CLIPConfig())
        m.load_state_dict(sd, strict=True)
        m = m.to(dev, torch.bfloat16).eval()
        px = synth.pixel_values(PAIRS, seed=4321).to(torch.bfloat16).to(dev)
        ids = synth.token_ids(PAIRS, seed=4322, full_length=True)[0].to(dev)

        def step():
            return m(input_ids=ids, pixel_values=px).logits_per_image

        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        # small-batch latency of the reference's default batch_size=8 (plip.py:95-97)
        lat = {}
        for b in (8, 32):
            pb, ib = px[:b], ids[:b]
            for _ in range(3):
                m(input_ids=ib, pixel_values=pb)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(10):
                m(input_ids=ib, pixel_values=pb)
            e1.record()
            torch.cuda.synchronize()
            lat[f"batch{b}_ms"] = e0.elapsed_time(e1) / 10
        del m
        torch.cuda.empty_cache()
        return {"impl": "transformers.CLIPModel.to(cuda, bfloat16), stock PyTorch kernels", "ms_per_step": ms,
                "pairs_per_s": PAIRS / ms * 1e3, **lat}
    except Exception as exc:  # noqa: BLE001
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}


class Timer:
    def __init__(self, dev, ws):
        self.dev, self.ws = dev, ws

    def barrier(self):
        if self.ws > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, keep_last=False):
        """barrier + sync, CUDA events on the launch stream around `steps` calls, barrier + sync, MAX over ranks (ms).
        With `keep_last`, returns (ms, what the last call returned)."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        out = None
        e0.record()
        for i in range(steps):
            out = None          # release the previous step's result before the next step runs, as if it were discarded
            out = fn(i)
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.ws > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return (ms, out) if keep_last else ms


DUMP_BYTES = 64 << 20          # --dump-outputs writes at most this much per run
DUMP_ARRAY_BYTES = 16 << 20    # a larger array is written as a seeded sample of its rows


def dump_outputs(ctx, arrays):
    """--dump-outputs DIR (rank 0): the arrays the timed path returned in its last step, as DIR/<name>.npy, so that two
    builds can be compared output for output.  Floating-point arrays are written as float32, integer ones as float64
    (exact).  An array above DUMP_ARRAY_BYTES keeps a sorted sample of its rows, drawn with a fixed seed from the row
    count alone (the same rows in every run); the row numbers go to DIR/<name>_rows.npy."""
    path = ctx["args"].dump_outputs
    if not path or ctx["rank"] != 0:
        return
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in arrays.items():
        t = t.detach()
        dtype = torch.float32 if t.is_floating_point() else torch.float64
        elem = 4 if dtype == torch.float32 else 8
        if t.numel() * elem > DUMP_ARRAY_BYTES:
            n = t.shape[0]
            k = max(1, DUMP_ARRAY_BYTES // (t[0].numel() * elem))
            rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False))
            np.save(os.path.join(path, f"{name}_rows.npy"), rows.astype(np.float64))
            total += rows.size * 8
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
        a = t.to(dtype).cpu().numpy()
        np.save(os.path.join(path, f"{name}.npy"), a)
        total += a.nbytes
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs wrote {total} bytes, more than {DUMP_BYTES}")


def run_ours(args):
    rank, local_rank, ws = _dist_env()
    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: plip_b200 has no CPU fallback"}))
        return 1
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if ws > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    torch.set_grad_enabled(False)
    torch.set_num_threads(max(1, min(32, usable_cores() // max(1, ws))))
    peaks = _peaks()

    configs = args.config.split(",")
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        sd, cpu = cpu_baseline_sample(configs[0])
        torch.set_num_threads(max(1, min(32, usable_cores() // max(1, ws))))
    else:
        from plip_b200 import synthetic
        sd = synthetic.make_state_dict(0)

    from plip_b200 import distributed as D
    from plip_b200._lib import lib
    from plip_b200.modeling import PlipCLIPModel
    # PLIP_BENCH_MB: experiment knob — engine micro-batch below the 1024-pair step (activations closer to L2 size)
    model = PlipCLIPModel(sd, device=dev, max_micro_batch=int(os.environ.get("PLIP_BENCH_MB", PAIRS)), operand_dtype=args.operands)
    ctx = {"args": args, "rank": rank, "ws": ws, "dev": dev, "peaks": peaks, "cpu": cpu, "sd": sd, "model": model,
           "eng": model.engine, "L": lib(), "sh": D.ShardedCLIP.from_engine(model.engine), "timer": Timer(dev, ws)}
    # several comma-separated configs share one process (one weight upload): one JSON line each — the driver's
    # default invocation names a single config and gets a single line
    rc = 0
    steps_arg = args.steps
    for name in configs:
        args.config = name
        args.steps = steps_arg if steps_arg is not None else {"pairs": 10, "cfg3": 5, "cfg4": 3, "cfg5": 2}[name]
        if name != configs[0]:
            ctx["cpu"] = None
        rc |= {"pairs": bench_pairs, "cfg3": bench_cfg3, "cfg4": bench_cfg4, "cfg5": bench_cfg5}[name](ctx)
        torch.cuda.empty_cache()
    return rc


def traffic_json():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
    except Exception:  # noqa: BLE001
        return None


def emit(ctx, value, unit, metric, ms_per_step, steps, scaling, clocks, e2e, launches, roofline, extra):
    args, ws = ctx["args"], ctx["ws"]
    line = {"metric": metric, "value": value, "unit": unit, "n_gpus": ws, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": args.operands, "data": "synthetic", "config": config_dict(args.config, ws), "clocks": clocks, "e2e": e2e,
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": ctx["cpu"], "extra": extra}
    print(json.dumps(line), flush=True)


# ---- default workload: 1024 x 1024 pairs per GPU per step ----------------------------------------------------------
def bench_pairs(ctx):
    from plip_b200 import synthetic as synth
    args, rank, ws, dev, peaks = ctx["args"], ctx["rank"], ctx["ws"], ctx["dev"], ctx["peaks"]
    model, eng, sh, L, timer = ctx["model"], ctx["eng"], ctx["sh"], ctx["L"], ctx["timer"]
    nsets = 2    # 2 alternating resident input sets (616 MB of pixels >> 126 MB L2)
    px = [synth.pixel_values(PAIRS, seed=1234 + 17 * rank + i).to(torch.bfloat16).to(dev) for i in range(nsets)]
    ids = [synth.token_ids(PAIRS, seed=1235 + 17 * rank + i, full_length=True)[0].to(dev) for i in range(nsets)]

    def step(i):
        return sh.clip_forward(px[i % nsets], ids[i % nsets])     # local images x the captions of all ranks

    sampler = ClockSampler(ctx["dev"].index) if rank == 0 else None   # started before the warm-up: nvidia-smi needs ~0.3 s
    for i in range(args.warmup):
        step(i)
    timer.barrier()
    launches0 = L.plip_launch_count()
    t_wall0 = time.time()
    ms, lpi = timer.timed(step, args.steps, keep_last=True)
    t_wall1 = time.time()
    launches = L.plip_launch_count() - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    dump_outputs(ctx, {"logits_per_image": lpi})
    del lpi
    ms_per_step = ms / args.steps
    value = PAIRS * ws * args.steps / (ms / 1e3)

    # ---- e2e: the product API on pinned HOST inputs (uint8 tiles + int64 ids in, logits out), every step
    tiles_h = [torch.from_numpy(synth.tiles_u8(PAIRS, seed=100 + rank + i)).pin_memory() for i in range(2)]
    ids_h = [synth.token_ids(PAIRS, seed=200 + rank + i, full_length=True)[0].pin_memory() for i in range(2)]
    out_h = [torch.empty(PAIRS, PAIRS * ws, dtype=torch.float32).pin_memory() for _ in range(2)]
    out_ev = [torch.cuda.Event() for _ in range(2)]

    def e2e_step(i):
        b = i & 1
        out_ev[b].synchronize()          # the logits of step i-2 have landed in this host buffer (the caller consumes them)
        if ws == 1:
            lg = model(input_ids=ids_h[b], pixel_values=tiles_h[b]).logits_per_image     # README.md:45-49 call
        else:
            px_d, up = eng.upload_async(tiles_h[b])                                      # pixels upload during the text tower
            txt_ids = ids_h[b].to(dev, non_blocking=True)
            lg = sh.clip_forward((_after(px_d, up, dev) for _ in range(1)), txt_ids)   # waited for only when the vision tower starts
        out_h[b].copy_(lg, non_blocking=True)                                             # D2H of this step's logits
        out_ev[b].record()

    for i in range(4):
        e2e_step(i)
    ms_e2e = timer.timed(e2e_step, args.steps)
    e2e = {"value": PAIRS * ws * args.steps / (ms_e2e / 1e3), "unit": "pairs/s",
           "h2d_bytes_per_step": PAIRS * 224 * 224 * 3 + PAIRS * 77 * 8, "d2h_bytes_per_step": PAIRS * PAIRS * ws * 4,
           "ms_per_step": ms_e2e / args.steps,
           "path": ("PlipCLIPModel.__call__(input_ids=<pinned host int64 [1024,77]>, pixel_values=<pinned host uint8 "
                    "[1024,224,224,3]>).logits_per_image -> pinned host buffer every step (two host buffers: step i's D2H overlaps the "
                    "launch of step i+1; the timed region ends with a full synchronise)"
                    if ws == 1 else
                    "ShardedCLIP.clip_forward on this rank's pinned host uint8 tiles + int64 ids (uploaded inside the step; "
                    "NCCL all-gather of the text embeddings) -> logits_per_image [1024, 1024*n_gpus] f32 to a pinned host "
                    "buffer every step (two host buffers; the timed region ends with a full synchronise)")}

    # ---- towers alone + in-step kernel profile (rank-local, after the timed regions)
    def tower(fn, reps=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ea.record()
        for _ in range(reps):
            fn()
        eb.record()
        torch.cuda.synchronize()
        return ea.elapsed_time(eb) / reps

    ms_v = tower(lambda: eng.encode_images(px[0]))
    ms_t = tower(lambda: eng.encode_text(ids[0]))
    if rank != 0:
        if ws > 1:
            # the other ranks keep the collective of the profiled steps company
            prof_steps = 2 + 3
            for i in range(prof_steps):
                step(i)
            torch.cuda.synchronize()
        return 0
    prof = in_step_profile(eng, lambda: step(0), peaks)
    roof, roof_worst = roofline_from_profile(prof, peaks, traffic_json())
    extra = {
        "step_tflops": (PAIRS * (FLOP_IMG + FLOP_TXT) + 2.0 * PAIRS * PAIRS * ws * 512) / (ms_per_step / 1e3) / 1e12,
        "roofline_worst": roof_worst,
        "kernels_in_step": prof,
        "vision_tower_1024_bf16": {"ms": ms_v, "img_per_s": PAIRS / ms_v * 1e3, "tflops": PAIRS * FLOP_IMG / ms_v / 1e9,
                                   "frac_of_burst_peak": PAIRS * FLOP_IMG / ms_v / 1e9 / peaks["bf16_tflops"],
                                   "frac_of_sustained_peak": PAIRS * FLOP_IMG / ms_v / 1e9 / peaks["bf16_tflops_sustained"]},
        "text_tower_1024x77": {"ms": ms_t, "captions_per_s": PAIRS / ms_t * 1e3, "tflops": PAIRS * FLOP_TXT / ms_t / 1e9,
                               "frac_of_sustained_peak": PAIRS * FLOP_TXT / ms_t / 1e9 / peaks["bf16_tflops_sustained"]},
    }
    extra["step_frac_of_sustained_peak"] = extra["step_tflops"] / peaks["bf16_tflops_sustained"]
    if ws == 1:
        # opt-in engine option, NOT the headline: the last layer's out_proj / LN2 / MLP on the pooled rows only
        # (identical embeddings, tests/test_gpu_model.py::test_last_layer_pruning_gives_the_same_embeddings)
        eng.set_last_layer_pruning(True)
        try:
            for i in range(3):
                step(i)
            ms_p = timer.timed(step, args.steps)
        finally:
            eng.set_last_layer_pruning(False)
        extra["last_layer_pruning_opt_in"] = {"value": PAIRS * args.steps / (ms_p / 1e3), "unit": "pairs/s",
                                              "ms_per_step": ms_p / args.steps,
                                              "what": "same step with Engine.set_last_layer_pruning(True); `value` above is measured without it"}
    if not args.quick:
        extra["kernels_alone_burst"] = kernel_bursts(eng, peaks, torch.cuda.current_stream().cuda_stream)
        extra.update(product_api_extras(ctx, tower))
        if not args.no_context:
            extra["stock_pytorch_bf16_same_gpu"] = stock_pytorch_context(ctx["sd"], dev)
    emit(ctx, value, "pairs/s", METRIC, ms_per_step, args.steps, "weak", clocks, e2e, launches, roof, extra)
    return 0


def _after(t, ev, dev):
    torch.cuda.current_stream(dev).wait_event(ev)
    return t


def product_api_extras(ctx, tower):
    """Other reference-facing calls, timed end to end from host objects (context next to the headline e2e)."""
    import PIL.Image
    from plip_b200 import synthetic as synth
    from plip_b200.plip import PLIP
    eng, model, dev = ctx["eng"], ctx["model"], ctx["dev"]
    out = {}
    try:
        tiles = synth.tiles_u8(PAIRS, seed=300)
        pil = [PIL.Image.fromarray(t) for t in tiles]
        p = PLIP("bench", model=model)
        if p is not None:
            p.encode_images(pil[:64], batch_size=32)
            t0 = time.perf_counter()
            emb = p.encode_images(pil, batch_size=32)
            dt = time.perf_counter() - t0
            out["PLIP.encode_images_1024_PIL_tiles"] = {"ms": dt * 1e3, "img_per_s": PAIRS / dt, "shape": list(emb.shape),
                                                        "note": "plip.py:31-53 call: List[PIL.Image] -> np.ndarray[1024,512]; "
                                                                "includes PIL->uint8 on the host, H2D, vision tower, D2H"}
        th = torch.from_numpy(tiles).pin_memory()
        eng.encode_images_host(th[:64])
        t0 = time.perf_counter()
        eng.encode_images_host(th)
        dt = time.perf_counter() - t0
        out["plip_encode_images_host_1024_u8"] = {"ms": dt * 1e3, "img_per_s": PAIRS / dt,
                                                  "note": "C ABI host-buffer call: pinned uint8 tiles in, [1024,512] f32 on the host out"}
        ids_h = synth.token_ids(PAIRS, seed=301, full_length=True)[0]
        eng.encode_text_host(ids_h[:64])
        t0 = time.perf_counter()
        eng.encode_text_host(ids_h)
        dt = time.perf_counter() - t0
        out["plip_encode_text_host_1024x77"] = {"ms": dt * 1e3, "captions_per_s": PAIRS / dt}
        ids_m, mask_m = synth.token_ids(4096, seed=302)                      # lengths U{8..77}: the bucketed host path
        eng.encode_text_host(ids_m[:256], mask_m[:256])
        t0 = time.perf_counter()
        eng.encode_text_host(ids_m, mask_m)
        dt_b = time.perf_counter() - t0
        ms_full = tower(lambda: eng.encode_text(ids_m.to(dev), mask_m.to(dev)), reps=2)
        out["text_length_buckets_4096_mixed"] = {"host_bucketed_ms": dt_b * 1e3, "device_full_length_ms": ms_full,
                                                 "note": "4096 captions with lengths U{8..77}: plip_encode_text_host (sorted into DP-chosen "
                                                         "length buckets, incl. H2D/D2H) vs the full-length 77-token device pass"}
        # small-batch latency (the reference's default batch_size = 8, plip.py:95-97): device inputs, synchronised
        lat = {}
        for b in (8, 32):
            pxb = synth.pixel_values(b, seed=9).to(torch.bfloat16).to(dev)
            idb = synth.token_ids(b, seed=10, full_length=True)[0].to(dev)
            for _ in range(3):
                model(input_ids=idb, pixel_values=pxb)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(20):
                model(input_ids=idb, pixel_values=pxb)
            torch.cuda.synchronize()
            lat[f"batch{b}_ms"] = (time.perf_counter() - t0) / 20 * 1e3
        out["small_batch_latency_forward"] = lat
    except Exception as exc:  # noqa: BLE001 - context only
        out["product_api_extras_error"] = f"{type(exc).__name__}: {exc}"[:300]
    return out


# ---- cfg3: 4096 images x 1024 captions, 1 GPU ----------------------------------------------------------------------
def bench_cfg3(ctx):
    from plip_b200 import synthetic as synth
    args, rank, ws, dev, peaks = ctx["args"], ctx["rank"], ctx["ws"], ctx["dev"], ctx["peaks"]
    model, eng, L, timer = ctx["model"], ctx["eng"], ctx["L"], ctx["timer"]
    n_img, n_txt = 4096, 1024
    px = torch.cat([synth.pixel_values(PAIRS, seed=1234 + i).to(torch.bfloat16) for i in range(4)]).to(dev)
    ids, mask = synth.token_ids(n_txt, full_length=True)
    ids = ids.to(dev)

    def step(i):
        return model(input_ids=ids, pixel_values=px)

    sampler = ClockSampler(dev.index) if rank == 0 else None
    for i in range(args.warmup):
        step(i)
    launches0 = L.plip_launch_count()
    t0 = time.time()
    ms, out = timer.timed(step, args.steps, keep_last=True)
    t1 = time.time()
    launches = L.plip_launch_count() - launches0
    clocks = sampler.stop(t0, t1) if sampler else None
    # logits_per_text is the transpose of logits_per_image
    dump_outputs(ctx, {k: out[k] for k in ("logits_per_image", "image_embeds", "text_embeds")})
    del out
    tiles_h = torch.from_numpy(synth.tiles_u8(n_img, seed=100)).pin_memory()
    ids_h = synth.token_ids(n_txt, seed=200, full_length=True)[0].pin_memory()
    out_h = torch.empty(n_img, n_txt, dtype=torch.float32).pin_memory()

    def e2e_step(i):
        out_h.copy_(model(input_ids=ids_h, pixel_values=tiles_h).logits_per_image, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for i in range(2):
        e2e_step(i)
    ms_e2e = timer.timed(e2e_step, args.steps)
    if rank != 0:
        return 0
    flop = n_img * FLOP_IMG + n_txt * FLOP_TXT + 2.0 * n_img * n_txt * 512
    prof = in_step_profile(eng, lambda: step(0), peaks, reps=2)
    roof, roof_worst = roofline_from_profile(prof, peaks, traffic_json())
    e2e = {"value": n_img * args.steps / (ms_e2e / 1e3), "unit": "pairs/s", "h2d_bytes_per_step": n_img * 150528 + n_txt * 77 * 8,
           "d2h_bytes_per_step": n_img * n_txt * 4, "ms_per_step": ms_e2e / args.steps,
           "path": "PlipCLIPModel.__call__ on pinned host uint8 tiles [4096,224,224,3] + int64 ids [1024,77] -> logits_per_image "
                   "[4096,1024] f32 in a pinned host buffer, synchronised every step"}
    extra = {"step_tflops": flop / (ms / args.steps / 1e3) / 1e12, "captions_per_s": n_txt * args.steps / (ms / 1e3),
             "pairs_definition": "pairs/s = images/s with N_txt / N_img = 1/4 (SURVEY.md §8d)",
             "roofline_worst": roof_worst, "kernels_in_step": prof}
    emit(ctx, n_img * args.steps / (ms / 1e3), "pairs/s", METRIC, ms / args.steps, args.steps, "strong", clocks, e2e, launches, roof, extra)
    return 0


# ---- cfg4 / cfg5: strong scaling over the GPUs of one box -----------------------------------------------------------
def _device_tiles(n, seed, dev, chunk=4096):
    """n synthetic uint8 tiles generated on the device (SURVEY.md §8d: seed 1234 + rank), in chunks."""
    g = torch.Generator(device=dev).manual_seed(seed)
    out = torch.empty(n, 224, 224, 3, dtype=torch.uint8, device=dev)
    for i in range(0, n, chunk):
        j = min(n, i + chunk)
        out[i:j] = torch.randint(0, 256, (j - i, 224, 224, 3), generator=g, device=dev, dtype=torch.uint8)
    return out


def bench_cfg4(ctx):
    from plip_b200 import distributed as D, synthetic as synth
    args, rank, ws, dev, peaks = ctx["args"], ctx["rank"], ctx["ws"], ctx["dev"], ctx["peaks"]
    eng, sh, L, timer = ctx["eng"], ctx["sh"], ctx["L"], ctx["timer"]
    n_total = args.tiles or 100000
    lo, hi = D.shard_range(n_total, rank, ws)
    n_local = hi - lo
    tiles = _device_tiles(n_local, 1234 + rank, dev)
    prompts = synth.token_ids(64, seed=1235)[0].to(dev)

    def step(i):
        return sh.zero_shot(tiles, prompts, n_total, gather_embeddings=True)

    sampler = ClockSampler(dev.index) if rank == 0 else None
    for i in range(min(args.warmup, 2)):
        step(i)
    launches0 = L.plip_launch_count()
    t0 = time.time()
    ms, (pred, logits, all_img) = timer.timed(step, args.steps, keep_last=True)
    t1 = time.time()
    launches = L.plip_launch_count() - launches0
    clocks = sampler.stop(t0, t1) if sampler else None
    dump_outputs(ctx, {"pred": pred, "logits": logits, "image_embeds": all_img})
    del pred, logits, all_img
    # e2e: the same flow fed from a pinned host ring of 2 x 1024 tiles, H2D of every micro-batch inside the timed region
    ring = [torch.from_numpy(synth.tiles_u8(PAIRS, seed=100 + rank + i)).pin_memory() for i in range(2)]
    pred_h = torch.empty(n_local, dtype=torch.int64).pin_memory()

    def host_chunks():
        for c, i in enumerate(range(0, n_local, PAIRS)):
            m = min(PAIRS, n_local - i)
            d, ev = eng.upload_async(ring[c & 1][:m])
            yield _after(d, ev, dev)

    def e2e_step(i):
        pred, _, _ = sh.zero_shot(host_chunks(), prompts.cpu().to(dev, non_blocking=True), n_total, gather_embeddings=True)
        pred_h.copy_(pred, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step(0)
    ms_e2e = timer.timed(e2e_step, args.steps)
    if rank != 0:
        return 0
    flop = n_total * FLOP_IMG + ws * 64 * FLOP_TXT
    metric, unit = metric_of("cfg4")
    e2e = {"value": n_total * args.steps / (ms_e2e / 1e3), "unit": unit, "h2d_bytes_per_step": n_local * 150528 + 64 * 77 * 8,
           "d2h_bytes_per_step": n_local * 8, "ms_per_step": ms_e2e / args.steps,
           "path": "ShardedCLIP.zero_shot over this rank's tiles uploaded micro-batch by micro-batch from a pinned host ring "
                   "(2 x 154 MB, re-read: a 15 GB pinned source would not change the copy rate), predictions back to pinned host"}
    extra = {"job_tflops": flop / (ms / args.steps / 1e3) / 1e12, "tiles_total": n_total, "tiles_per_rank": n_local,
             "outputs": "pred [n_local], logits [n_local,64], all-gathered image_embeds [n_total,512] on every rank"}
    emit(ctx, n_total * args.steps / (ms / 1e3), unit, metric, ms / args.steps, args.steps, "strong", clocks, e2e, launches, None, extra)
    return 0


def bench_cfg5(ctx):
    from plip_b200 import distributed as D, synthetic as synth
    args, rank, ws, dev, peaks = ctx["args"], ctx["rank"], ctx["ws"], ctx["dev"], ctx["peaks"]
    eng, sh, L, timer = ctx["eng"], ctx["sh"], ctx["L"], ctx["timer"]
    n_gal = args.tiles or 1000000
    n_q = args.queries or 10000
    lo, hi = D.shard_range(n_gal, rank, ws)
    n_local = hi - lo
    qlo, qhi = D.shard_range(n_q, rank, ws)
    pool_n = 8192
    pool = _device_tiles(pool_n, 1234 + rank, dev)
    q_ids = synth.token_ids(n_q, seed=1235)[0][qlo:qhi].to(dev)

    def gallery_chunks():
        for i in range(0, n_local, PAIRS):
            m = min(PAIRS, n_local - i)
            s = (i % pool_n)
            yield pool[s:s + m] if s + m <= pool_n else torch.cat([pool[s:], pool[:s + m - pool_n]])

    state = {}

    def step(i):
        block, gal, q_all = sh.retrieval(gallery_chunks(), q_ids, n_q)      # [n_local, n_q] f32 row block
        state["gal"], state["q_all"] = gal, q_all
        return block

    sampler = ClockSampler(dev.index) if rank == 0 else None
    for i in range(min(args.warmup, 1)):
        step(i)
    launches0 = L.plip_launch_count()
    t0 = time.time()
    ms, block = timer.timed(step, args.steps, keep_last=True)
    t1 = time.time()
    launches = L.plip_launch_count() - launches0
    clocks = sampler.stop(t0, t1) if sampler else None
    gal, q_all = state["gal"], state["q_all"]
    dump_outputs(ctx, {"similarity": block, "gallery_embeds": gal, "query_embeds": q_all})
    del block
    # the similarity block and the fused top-k head alone
    sh.similarity(gal, q_all, sh.logit_scale_exp)
    sh.retrieval_topk(gal, q_all, 50, n_gal)                      # untimed first calls: scratch growth, lazy module loading
    ms_sim = timer.timed(lambda i: sh.similarity(gal, q_all, sh.logit_scale_exp), 3) / 3
    ms_topk = timer.timed(lambda i: sh.retrieval_topk(gal, q_all, 50, n_gal), 3) / 3
    # e2e: gallery micro-batches uploaded from a pinned host ring inside the timed region; top-50 per query returned
    ring = [torch.from_numpy(synth.tiles_u8(PAIRS, seed=100 + rank + i)).pin_memory() for i in range(2)]
    top_h = torch.empty(n_q, 50, dtype=torch.int64).pin_memory()
    q_ids_h = q_ids.cpu().pin_memory()

    def host_chunks():
        for c, i in enumerate(range(0, n_local, PAIRS)):
            m = min(PAIRS, n_local - i)
            d, ev = eng.upload_async(ring[c & 1][:m])
            yield _after(d, ev, dev)

    def e2e_step(i):
        block, g, qa = sh.retrieval(host_chunks(), q_ids_h.to(dev, non_blocking=True), n_q)
        idx, _ = sh.retrieval_topk(g, qa, 50, n_gal)
        top_h.copy_(idx, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    e2e_step(0)
    ms_e2e = timer.timed(e2e_step, max(1, args.steps // 2))
    if rank != 0:
        return 0
    metric, unit = metric_of("cfg5")
    flop = n_gal * FLOP_IMG + n_q * FLOP_TXT + 2.0 * n_gal * n_q * 512
    sim_flop = 2.0 * n_local * n_q * 512
    e2e = {"value": n_gal * max(1, args.steps // 2) / (ms_e2e / 1e3), "unit": unit,
           "h2d_bytes_per_step": n_local * 150528 + (qhi - qlo) * 77 * 8, "d2h_bytes_per_step": n_q * 50 * 8,
           "ms_per_step": ms_e2e / max(1, args.steps // 2),
           "path": "ShardedCLIP.retrieval + retrieval_topk(k=50): gallery micro-batches uploaded from a pinned host ring, "
                   "query ids from pinned host, global top-50 image indices per query back to pinned host"}
    extra = {"job_tflops": flop / (ms / args.steps / 1e3) / 1e12, "gallery_total": n_gal, "gallery_per_rank": n_local, "queries": n_q,
             "similarity_block": {"shape": [n_local, n_q], "ms": ms_sim, "tflops_fp32": sim_flop / ms_sim / 1e9,
                                  "write_GBps": n_local * n_q * 4 / ms_sim / 1e6,
                                  "frac_of_hbm_peak": n_local * n_q * 4 / ms_sim / 1e6 / peaks["hbm_gbs"]},
             "fused_topk50_merge": {"ms": ms_topk, "note": "top-50 of all queries over this rank's gallery rows (tensor-core score chunks + "
                                                           "row merge) + all-gather of candidates + merge (retrieval.py:13-16 semantics)"}}
    emit(ctx, n_gal * args.steps / (ms / 1e3), unit, metric, ms / args.steps, args.steps, "strong", clocks, e2e, launches, None, extra)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="pairs", help="pairs (default) | cfg3 | cfg4 | cfg5, or a comma-separated list")
    ap.add_argument("--tiles", type=int, default=0, help="cfg4 / cfg5: override the total tile count (default 100k / 1M)")
    ap.add_argument("--queries", type=int, default=0, help="cfg5: override the query count (default 10k)")
    ap.add_argument("--operands", default="bf16", choices=["bf16", "fp16"],
                    help="16-bit format of the GEMM / attention operands (default bf16 = BASELINE.json's dtype)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-context", action="store_true", help="skip the stock-PyTorch-on-GPU context measurement")
    ap.add_argument("--quick", action="store_true", help="skip the extras (kernels alone, product-API extras, context)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned in its last step (rank 0) as DIR/<name>.npy, at most 64 MB; "
                         "one config, --impl ours")
    args = ap.parse_args()
    for c in args.config.split(","):
        if c not in WORKLOADS:
            ap.error(f"unknown config {c!r}")
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or "," in args.config):
        ap.error("--dump-outputs needs --impl ours and a single config")
    if args.impl == "reference":
        args.config = args.config.split(",")[0]
        if args.steps is None:
            args.steps = 5
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rc = run_reference(args) if args.impl == "reference" else run_ours(args)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()
    sys.exit(rc)


if __name__ == "__main__":
    main()
