#!/usr/bin/env python
"""bench.py -- BASELINE.json's headline metric: ViT-L/14-adapter 588x588 train images/s.

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA kernels)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the reference's own modules (oracle/_ref)
    torchrun --nproc-per-node N bench.py --gpus N ...        # N > 1, one rank per GPU over NCCL

One "step" = one training iteration of the reference's train() loop body (train.py:268-441) on one
batch of 12 synthetic 588x588 frames per GPU: encoder (24-block ViT-L/14 taps + interleaved
backbone/adapter pass) -> decoder -> dice loss -> backward through everything -> gradient
all-reduce (N > 1) -> SGD.  Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "ViT-L/14-adapter 588^2 train images/s"
UNIT = "images/s"


def ncu_traffic(key):
    """DRAM bytes of one representative launch of the kernel family `key`, from the committed ncu capture
    (profiles/ncu_traffic.json); None when there is no capture."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[key]
        return {"dram_bytes_per_launch": t["dram_bytes"], "algorithmic_bytes": t["algorithmic_bytes"],
                "launch": t["launch"], "source": t["source"]}
    except Exception:
        return None


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


class SpanProfiler:
    """CUDA-event pairs around every libasis_b200 op of one step (launching stream)."""

    def __init__(self):
        self.spans = []

    def begin(self, name, work, unit, detail=None):
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        return (name, work, unit, e0, e1, detail)

    def end(self, tok):
        tok[4].record()
        self.spans.append(tok)

    def summary(self):
        torch.cuda.synchronize()
        agg = {}
        self.detail = {}
        for name, work, unit, e0, e1, detail in self.spans:
            a = agg.setdefault(name, {"n": 0, "ms": 0.0, "work": 0.0, "unit": unit})
            ms = e0.elapsed_time(e1)
            a["n"] += 1
            a["ms"] += ms
            a["work"] += work
            if detail is not None:
                d = self.detail.setdefault((name, detail), {"n": 0, "ms": 0.0, "work": 0.0})
                d["n"] += 1
                d["ms"] += ms
                d["work"] += work
        return agg

    def detail_table(self):
        """per-shape breakdown (call after summary()): markdown rows sorted by time"""
        rows = sorted(self.detail.items(), key=lambda kv: -kv[1]["ms"])
        out = ["| ms | launches | us/launch | TFLOP/s | op | shape |", "|---:|---:|---:|---:|---|---|"]
        for (name, detail), d in rows:
            out.append(f"| {d['ms']:.2f} | {d['n']} | {1e3 * d['ms'] / d['n']:.1f} | {d['work'] / d['ms'] / 1e9:.0f} | {name} | {detail} |")
        return "\n".join(out)


def synth_batch(B, size, n_cls, seed):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 3, size, size, generator=g)                 # un-normalised [0,1) pixels (tools/dataset.py:159)
    tgt = torch.randint(0, n_cls, (B, size, size), generator=g)
    if torch.cuda.is_available():
        return img.pin_memory(), tgt.pin_memory()
    return img, tgt


# --------------------------------------------------------------------------------------------------
def cpu_reference_step(sds, img, target, heads):
    """The oracle port of the reference path on the host cores: fwd + bwd of the same step."""
    from oracle import encoder as o_enc
    params = []
    for sd in sds.values():
        for v in sd.values():
            if v.is_floating_point() and v.requires_grad:
                v.grad = None
                params.append(v)
    res = o_enc.adapter_encoder(sds["vit"], sds["spm"], sds["inj"], sds["ext"], img, heads)
    logits = o_enc.feature_decoder(sds["dec"], res["feat"])
    logits = torch.nn.functional.interpolate(logits, size=target.shape[-2:], mode="bilinear")
    loss = o_enc.dice_loss(torch.softmax(logits, 1), target)
    loss.backward()
    return float(loss)


def build_cpu_state(arch, seed=0):
    """Random-init parameters with the reference's names, on the CPU (plain tensors)."""
    import adaptersis_b200 as asis
    torch.manual_seed(seed)
    with torch.device("cpu"):
        enc = asis.AdapterEncoder(arch=arch)
        C = enc.model.embed_dim
        dec = asis.FeatureDecoder(embed_dim=C, num_classes=2, features=[C, 512, 256, 128, 64])
    sds = {"vit": enc.model.state_dict(), "spm": enc.backbone_encoder.state_dict(), "inj": enc.cross_vit.state_dict(),
           "ext": enc.cross_cnn.state_dict(), "dec": dec.state_dict()}
    out = {}
    for k, sd in sds.items():
        out[k] = {n: (v.detach().clone().requires_grad_(True) if v.is_floating_point() and "running" not in n else v)
                  for n, v in sd.items()}
    return out, enc.model.num_heads


ADAPTER_HEADS = {"vit_small": 6, "vit_base": 12, "vit_large": 8}     # train.py:86-110 uses 8 with ViT-L


def make_cpu_step(arch):
    """The CPU leg's step function: the reference's OWN modules when oracle/make_ref.sh has staged them under
    oracle/_ref/ (kind "reference"), else the oracle port (kind "port").  Returns (step(img, tgt) -> loss, kind, what)."""
    from oracle import ref_step
    if ref_step.available() and not os.environ.get("ASIS_CPU_PORT"):
        rs = ref_step.ReferenceStep(arch, adapter_heads=ADAPTER_HEADS.get(arch, 8))
        return rs.step, "reference", ("the reference's own unmodified PyTorch modules (oracle/_ref: MSDeformAttn via "
                                      "ms_deform_attn_core_pytorch/grid_sample, CAViT, CACNN, DINOv2 blocks with the naive "
                                      "attention path, FeatureEncoder, FeatureDecoder, DC loss)")
    sds, heads = build_cpu_state(arch)
    return (lambda img, tgt: cpu_reference_step(sds, img, tgt, heads)), "port", \
        "oracle port (pure PyTorch fp32 restatement of the reference modules)"


def run_reference(args, rank):
    if rank != 0:
        return
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    step_fn, kind, what = make_cpu_step(args.arch)
    img, tgt = synth_batch(1, args.imsize, 2, 1234)
    budget_s = float(os.environ.get("ASIS_REF_BUDGET_S", "170"))
    t_begin = time.perf_counter()
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        step_fn(img, tgt)
        dt_ = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt_)
        if time.perf_counter() - t_begin > budget_s and times:       # bounded run: stop early, report what was timed
            break
    ms = 1e3 * sum(times) / len(times)
    val = 1.0 / (ms / 1e3)
    sample = (f"{len(times)} timed step(s) of 1 image each (of the 12-image batch), full {args.arch} /14 + adapters + decoder "
              f"fwd+bwd, {what}, {ncores} threads")
    line = {"impl": "reference", "metric": METRIC, "value": round(val, 5), "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(times), "warmup": args.warmup, "ms_per_step": round(ms, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args, 1, "cpu"),
            "cpu_baseline": {"value": round(val, 5), "unit": UNIT, "cores": ncores, "kind": kind, "sample": sample},
            "e2e": {"value": round(val, 5), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def config_dict(args, per_gpu_batch, where):
    cfg = {"vit_large": "config[2]", "vit_base": "config[1]"}.get(args.arch, "(not a BASELINE config)")
    return {"workload": f"{cfg}: {args.arch.replace('_', '-')}/14 + adapter (n_last_blocks 4) train step, imsize "
                        f"{args.imsize}, batch {per_gpu_batch}/GPU",
            "arch": args.arch, "imsize": args.imsize, "tokens": (args.imsize // 14) ** 2 + 1,
            "global_batch": per_gpu_batch * max(1, args.gpus if where != "cpu" else 1), "parallelism": f"dp{args.gpus}",
            "backward": "full (backbone dgrad+wgrad, adapters, SPM, decoder); taps pass forward-only as in the reference",
            "optimizer": "SGD(momentum 0.99, wd 3e-5) on all parameters",
            "launch": "whole step replayed as one CUDA graph" if getattr(args, "graph_used", False) else "eager launches",
            "cache": "per-step working set (>15 GB of activations) >> 126 MB L2; no explicit flush needed",
            **({"gradient_exchange": getattr(args, "dp_schedule", "")} if where != "cpu" and args.gpus > 1 else {})}


DUMP_SAMPLE = 4 << 20          # parameter values written by --dump-outputs (float32: 16 MB)


def dump_outputs(out_dir, ts, loss):
    """What the last timed step handed back to its caller: the loss and the parameters the SGD update wrote, as
    loss.npy (float64), param_norms.npy (float64 L2 norm of every parameter, in ts.parameters() order) and
    param_sample.npy (float32, the same DUMP_SAMPLE positions of the concatenated parameters every run)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    params = [p.detach() for p in ts.parameters()]
    np.save(os.path.join(out_dir, "loss.npy"), np.array([float(loss.detach())], dtype=np.float64))
    np.save(os.path.join(out_dir, "param_norms.npy"), torch.stack([p.double().norm() for p in params]).cpu().numpy())
    flat = torch.cat([p.reshape(-1).float() for p in params])
    idx = torch.randint(0, flat.numel(), (min(DUMP_SAMPLE, flat.numel()),), generator=torch.Generator().manual_seed(0))
    np.save(os.path.join(out_dir, "param_sample.npy"), flat[idx.sort().values.to(flat.device)].cpu().numpy())


# --------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import adaptersis_b200 as asis
    from adaptersis_b200 import _lib, kernels
    from adaptersis_b200.trainer import TrainStep

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.manual_seed(0)
    B = args.batch
    ts = TrainStep(arch=args.arch, device=dev, precision=args.precision, train_backbone=not args.frozen_backbone)
    batches = [synth_batch(B, args.imsize, 2, 100 * rank + i) for i in range(2)]
    dev_batches = [(a.to(dev), b.to(dev)) for a, b in batches]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        ts.step_device(*dev_batches[i % 2])
    barrier()
    # whole-step CUDA graph; with N > 1 the NCCL side stream of the bucketed all-reduce joins the capture
    # (measured at N = 2: 139.2 vs 141.1 ms; ASIS_GRAPH_DP=0 turns it off)
    use_graph = not args.no_graph and (world == 1 or os.environ.get("ASIS_GRAPH_DP", "1") != "0")
    args.graph_used = use_graph
    args.dp_schedule = f"NCCL all-reduce (AVG, fp32, {ts.reducer.bucket_bytes >> 20} MB buckets) " + \
        ("overlapped with backward on a side stream" if ts.reducer.overlap else
         "after backward, back to back; gradients stay views into the reduced buckets")
    if use_graph:
        ts.capture(*dev_batches[0])
        for i in range(2):                                   # warm replays
            ts.step_device(*dev_batches[i % 2])
        barrier()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    # process-wide start/end range (backward runs on autograd's thread, outside any push/pop range of this
    # one):  ncu --nvtx --nvtx-include "asis_timed"  profiles only the timed steps
    rng = torch.cuda.nvtx.range_start("asis_timed")
    for i in range(args.steps):
        loss = ts.step_device(*dev_batches[i % 2])
    torch.cuda.nvtx.range_end(rng)
    e1.record()
    barrier()
    launches = _lib.launch_count() - n0 + args.steps * ts.graph_launches     # eager launches + kernel nodes replayed
    t_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ts, loss)

    if args.only_timed:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": round(B * world * args.steps / (t_ms * 1e-3), 3), "unit": UNIT,
                              "ms_per_step": round(t_ms / args.steps, 2), "gpu_launches": int(launches),
                              "note": "--only-timed run (for ncu): no e2e / profile / cpu legs"}), flush=True)
        return
    # end to end: pinned host batch in, python float out, every step
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for i in range(args.steps):
        lv = ts.step(*batches[i % 2])
    e3.record()
    barrier()
    t_e2e_ms = e2.elapsed_time(e3)

    tt = torch.tensor([t_ms, t_e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms, t_e2e_ms = float(tt[0]), float(tt[1])

    # one extra, un-timed step with per-op CUDA events -> roofline of the dominant kernel
    # (every rank runs it -- the step contains collectives -- only rank 0 records)
    prof = SpanProfiler()
    if rank == 0:
        kernels.set_profiler(prof)
    torch.cuda.synchronize()
    p0 = torch.cuda.Event(enable_timing=True)
    p1 = torch.cuda.Event(enable_timing=True)
    p0.record()
    ts.step_device(*dev_batches[0], eager=True)             # (events between launches: not through the graph)
    p1.record()
    kernels.set_profiler(None)
    barrier()
    if rank != 0:
        return
    agg = prof.summary()
    prof_step_ms = p0.elapsed_time(p1)
    step_ms = t_ms / args.steps        # shares are taken against the TIMED step (the profiled one carries an event pair per op)
    pk, pk_src = peaks()

    def tensor_roof(names, peak_tf):
        ms = sum(agg[n]["ms"] for n in names if n in agg)
        work = sum(agg[n]["work"] for n in names if n in agg)
        n = sum(agg[n]["n"] for n in names if n in agg)
        if ms <= 0:
            return None
        ach = work / (ms * 1e-3) / 1e12
        return {"bound": "tensor", "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s",
                "frac": round(ach / peak_tf, 3), "traffic": None, "launches": n, "ms_in_step": round(ms, 2),
                "share_of_step": round(ms / step_ms, 3), "peak_source": f"{pk_src} (sustained: timed inside a long step)"}

    def hbm_roof(names):
        ms = sum(agg[n]["ms"] for n in names if n in agg)
        work = sum(agg[n]["work"] for n in names if n in agg)
        n = sum(agg[n]["n"] for n in names if n in agg)
        if ms <= 0:
            return None
        ach = work / (ms * 1e-3) / 1e9
        return {"bound": "hbm", "achieved": round(ach, 1), "peak": pk["hbm_gbs"], "unit": "GB/s",
                "frac": round(ach / pk["hbm_gbs"], 3), "traffic": None, "launches": n, "ms_in_step": round(ms, 2),
                "share_of_step": round(ms / step_ms, 3), "peak_source": pk_src}

    peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    roof = tensor_roof(["gemm_bf16"], peak_tf) or tensor_roof(["gemm_f32"], peak_tf)
    if roof is not None and "gemm_bf16" in agg:
        tr = ncu_traffic("gemm_bf16")
        if tr is not None:      # bytes of ONE captured launch (dram__bytes_read + write), with its algorithmic bytes beside it
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_detail"] = tr
    table = {k: {"n": v["n"], "ms": round(v["ms"], 3)} for k, v in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])}
    print("[bench] per-op time inside one profiled step (ms):", json.dumps(table), file=sys.stderr)
    print(f"[bench] profiled step {prof_step_ms:.1f} ms; timed step {t_ms / args.steps:.1f} ms", file=sys.stderr)
    if args.detail:
        print("[bench] per-shape breakdown of the profiled step:\n" + prof.detail_table(), file=sys.stderr)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            ncores = os.cpu_count() or 1
            torch.set_num_threads(ncores)
            step_fn, kind, what = make_cpu_step(args.arch)
            img, tgt = synth_batch(1, args.imsize, 2, 1234)
            step_fn(img, tgt)                                   # 1 warm-up (BASELINE.md section 4)
            ts_ = []
            for _ in range(3):
                t0 = time.perf_counter()
                step_fn(img, tgt)
                ts_.append(time.perf_counter() - t0)
            cpu = {"value": round(1.0 / min(ts_), 5), "unit": UNIT, "cores": ncores, "kind": kind,
                   "sample": f"1 image (of the 12-image batch) per step, 1 warm-up + min of 3 fwd+bwd steps "
                             f"({', '.join(f'{t:.2f}' for t in ts_)} s) through {what}, all host threads"}
        except Exception as ex:  # pragma: no cover
            cpu = {"value": None, "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex!r}"}

    # BASELINE.json's second metric: MSDeformAttn achieved HBM GB/s (fwd and bwd) on algorithmic bytes, at the two real
    # shapes of the step and two points of the config[4] sweep (M=16, D=64), fp32 and the bf16-value variant
    msda = None
    if world == 1 and not args.no_msda:
        try:
            from tools.msda_bench import REAL_CASES, run_cases
            extra = [("sweep_g36_Lq1764", 12, 1764, 16, 64, [(72, 72), (36, 36), (18, 18)], 4),
                     ("sweep_g36_Lq6949", 12, 6949, 16, 64, [(72, 72), (36, 36), (18, 18)], 4)]
            rows = run_cases(REAL_CASES + extra, dev, pk["hbm_gbs"], iters=7)
            msda = {"unit": "GB/s", "peak": pk["hbm_gbs"], "peak_source": pk_src, "bytes": "algorithmic (SURVEY.md 8d), "
                    "value counted once and only where samples can touch it", "timing": "median of 7, L2 flushed "
                    "between iterations, CUDA events", "cases": rows}
        except Exception as ex:  # pragma: no cover
            msda = {"failed": repr(ex)}

    imgs = B * world * args.steps
    h2d = sum(t.numel() * t.element_size() for t in batches[0])
    line = {"metric": METRIC, "value": round(imgs / (t_ms * 1e-3), 3), "unit": UNIT, "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t_ms / args.steps, 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": config_dict(args, B, "gpu"),
            "e2e": {"value": round(imgs / (t_e2e_ms * 1e-3), 3), "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(t_e2e_ms / args.steps, 2)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof,
            "roofline_attention": tensor_roof(["attn_fwd", "attn_bwd"], peak_tf),
            "roofline_msda": hbm_roof(["msda_fwd", "msda_bwd"]),
            # the 3x3 convolutions of the stem / decoder run on the same tcgen05 kernel as implicit GEMMs; at 64-128 channels
            # they are bound by their maps' bytes, not by the tensor pipe, and are kept out of `roofline` (the Linear GEMMs)
            "roofline_conv": tensor_roof(["conv_bf16"], peak_tf),
            "msda": msda, "cpu_baseline": cpu, "last_loss": lv}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--arch", default="vit_large")
    ap.add_argument("--batch", type=int, default=12)
    ap.add_argument("--imsize", type=int, default=588)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--frozen-backbone", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-msda", action="store_true", help="skip the MSDeformAttn GB/s record")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying the step's CUDA graph")
    ap.add_argument("--detail", action="store_true", help="print the per-shape GEMM breakdown of the profiled step")
    ap.add_argument("--only-timed", action="store_true", help="warm-up + timed loop only (used under ncu)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the loss and parameters of the last timed step as "
                    "DIR/*.npy, to compare two builds on identical inputs")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
