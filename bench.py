#!/usr/bin/env python
"""Headline benchmark: htdemucs audio-seconds separated per second on N B200s.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the host CPU
    python bench.py --gpus 1 ... --dump-outputs DIR          # also store what the last timed step computed

Workload (BASELINE.json configs[2]): htdemucs (random-init, 4 stems, 41.98 M parameters), one
synthetic stereo 44.1 kHz track of 64 x 7.8 s segments (overlap 0.25, shifts=0) run through
``apply_model``: segments are batched through the kernel engine, overlap-added on the device, and --
for N > 1 -- sharded 64/N per rank in contiguous blocks (strong scaling) with an exchange of the
overlap slabs between neighbours; every rank hands the samples it produced to the host.  A "step" is
one ``apply_model`` pass over the whole track.  ``weak`` (N > 1) is the same call on a track of 64
segments PER GPU.

Prints ONE JSON line (rank 0).  ``value`` = track seconds / device time with the track resident
in HBM; ``e2e`` = the same through the public API from pinned host memory and back.  The default
arithmetic ("strict") is the one that meets the north_star's fp32/TF32 tolerance (per-stem rel-L2
<= 1e-4); ``parity`` holds the measured figure of the run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEGMENTS = 64               # BASELINE configs[2]
CPU_SAMPLE_SEGMENTS = 8     # bounded sample of the same track for the CPU arms (about 47 s of audio)
SEG_LEN = 343980            # int(39/5 * 44100)
STRIDE = 257985             # int(0.75 * SEG_LEN)
SR = 44100
METRIC = "htdemucs audio-seconds separated per second"
UNIT = "audio-s/s"


def synth_track(length: int, seed: int = 1234):
    import torch
    g = torch.Generator().manual_seed(seed)
    return 0.1 * torch.randn(1, 2, length, generator=g)


TEN_MIN = 600 * SR           # 26 460 000 samples -> 103 segments per pass
# name -> (label, track length, shifts, default mode); the first is the headline (BASELINE configs[2])
WORKLOADS = {
    "configs2": (f"htdemucs 4-stem random-init, one track of {SEGMENTS}x7.8s segments (BASELINE configs[2]), "
                 f"apply_model overlap=0.25 shifts=0, segments sharded {SEGMENTS}/N per GPU", SEGMENTS * STRIDE, 0, "strict"),
    "6s_10min": ("htdemucs_6s 6-stem random-init, 10-minute track, apply_model overlap=0.25 shifts=2 (BASELINE configs[3]): "
                 "2 x 103 segment forwards sharded across the GPUs", TEN_MIN, 2, "strict"),
    "ft_10min": ("htdemucs_ft bag of 4 per-source htdemucs models (random-init), 10-minute track, overlap=0.25 shifts=0, bf16 mode "
                 "(BASELINE configs[4]): 4 x 103 segment forwards, every member's segments sharded across the GPUs", TEN_MIN, 0, "bf16"),
}


def workload_config(n_gpus: int, mode: str, batch: int, name: str = "configs2") -> dict:
    label, length, shifts, _ = WORKLOADS[name]
    return {"workload": label, "name": name, "segments": -(-length // STRIDE) * max(shifts, 1) * (4 if name == "ft_10min" else 1),
            "track_seconds": length / SR, "forward_batch": batch, "mode": mode, "parallelism": f"segments sharded x{n_gpus}",
            "l2": "inputs larger than L2 (>= 132 MB track, multi-GB activations per step)"}


def build_workload(name: str, mode: str, dev):
    """(model for demucs_b200, [(weights, cfg)] + bag weights for the oracle)"""
    import demucs_b200 as D
    from demucs_b200.config import htdemucs_config, htdemucs_6s_config
    from demucs_b200.weights import init_weights
    if name == "6s_10min":
        cfg = htdemucs_6s_config()
        return D.HTDemucs.from_config(cfg, init_seed=0, mode=mode).to(dev), (init_weights(cfg, 0), cfg), None
    if name == "ft_10min":
        cfg = htdemucs_config()
        ident = [[1.0 if s == m else 0.0 for s in range(4)] for m in range(4)]     # remote/htdemucs_ft.yaml
        models = [D.HTDemucs.from_config(cfg, init_seed=10 + m, mode=mode).to(dev) for m in range(4)]
        return D.BagOfModels(models, ident), [(init_weights(cfg, 10 + m), cfg) for m in range(4)], ident
    cfg = htdemucs_config()
    return D.htdemucs(mode=mode).to(dev), (init_weights(cfg, 0), cfg), None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.thread.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        busy = [c for c in sm if c >= 0.5 * (mx[0] if mx else 1)] or sm
        return {"sm_mhz": busy[len(busy) // 2] if busy else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_traffic(label: str, mode: str):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) and tensor-pipe activity of the kernels
    behind a profile label, from the committed ncu pass over one 16-segment forward in this mode
    (profiles/r02_ncu_forward_b16_<mode>.json, made by tools/ncu_forward_table.py).  None when absent."""
    path = os.path.join(ROOT, "profiles", f"r02_ncu_forward_b16_{mode}.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        table = json.load(f)["kernels"]
    if label.startswith("conv_gemm_tc<"):
        tbk, tbn = label[len("conv_gemm_tc<"):-1].split(",")     # label = kernel template <TBK,TBN>
        rows = [r for r in table if r["kernel"].replace(" ", "").startswith(f"conv_gemm_tc_persist_kernel<{tbk},{tbn},")]
    else:
        key = {"attention_tc": "attention_"}.get(label, label)
        rows = [r for r in table if r["kernel"].startswith(key)]
    if not rows:
        return None
    n = sum(r["launches"] for r in rows)
    ms = sum(r["ms"] for r in rows)
    return {"bytes_per_launch": sum(r["dram_mb"] for r in rows) * 1e6 / n, "launches": n,
            "tensor_pipe_active": sum(r["tensor_pipe_active"] * r["ms"] for r in rows) / ms,
            "source": os.path.relpath(path, ROOT)}


DUMP_BYTES = 60 << 20      # --dump-outputs: data in all; with the .npy headers still under 64 MB (10^6 or 2^20 bytes)
DUMP_WINDOW = 4096         # samples per window of a sampled output


def dump_outputs(outdir: str, arrays: dict) -> None:
    """Write each array of the last timed step as ``<outdir>/<name>.npy`` in float32.  An array larger than its share of
    DUMP_BYTES keeps the windows of DUMP_WINDOW samples along its last (time) axis at fixed, seeded positions, the same
    in every run with the same arguments, so that two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(outdir, exist_ok=True)
    share = DUMP_BYTES // len(arrays)
    for name, x in arrays.items():
        x = x.detach()
        length = x.shape[-1]
        if 4 * x.numel() > share:
            windows = length // DUMP_WINDOW
            keep = max(1, min(windows, share // (4 * (x.numel() // length) * DUMP_WINDOW)))
            starts = torch.randperm(windows, generator=torch.Generator().manual_seed(0))[:keep].sort().values
            idx = (starts[:, None] * DUMP_WINDOW + torch.arange(DUMP_WINDOW)).reshape(-1)
            x = x[..., idx.to(x.device)]
        np.save(os.path.join(outdir, f"{name}.npy"), x.float().cpu().numpy())


def measured_peaks() -> dict:
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops_sustained"], "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1400.0, "source": "fallback"}


# ------------------------------------------------------------------------------------------ CPU arms
def cpu_apply_seconds(length: int, reps: int, threads: int, want_output: bool = False):
    """Time the reference algorithm's apply_model on the host CPU: the unmodified reference when
    its tree is present, otherwise the oracle port."""
    import torch
    from oracle import refload
    from demucs_b200.config import htdemucs_config
    from demucs_b200.weights import init_weights
    torch.set_num_threads(threads)
    cfg = htdemucs_config()
    W = init_weights(cfg, 0)
    mix = synth_track(SEGMENTS * STRIDE)[..., :length].contiguous()     # a prefix of the GPU arm's own track
    if refload.available():
        ref = refload.load()
        model = refload.build_reference_model(cfg, W)
        kind = "reference"

        def run():
            return ref.apply_model(model, mix, shifts=0, split=True, overlap=0.25, device="cpu")
    else:
        from oracle.apply_oracle import apply_model_oracle
        kind = "port"

        def run():
            return apply_model_oracle((W, cfg), mix, shifts=0, split=True, overlap=0.25)
    times, out = [], None
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            out = run()
            times.append(time.perf_counter() - t0)
    if want_output:
        return times, kind, (mix, out)
    return times, kind


def reference_arm(args) -> None:
    """--impl reference: the reference's CPU implementation of the path on this host's cores, on a bounded sample
    (the first CPU_SAMPLE_SEGMENTS segments) of the same 64-segment track the GPU arm separates."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    length = CPU_SAMPLE_SEGMENTS * STRIDE
    times, kind, (_, out) = cpu_apply_seconds(length, args.warmup + args.steps, threads, want_output=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stems": out})
    timed = times[args.warmup:]
    sec = sum(timed) / len(timed)
    value = (length / SR) / sec
    sample = (f"{len(timed)} x apply_model on the first {CPU_SAMPLE_SEGMENTS} segments ({length / SR:.1f} s) of the bench "
              f"track, {threads} threads, torch CPU fp32")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, "cpu-fp32", 1),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ GPU arm
DTYPE = {"strict": "f32 (bf16 hi/lo split operands, 3 tcgen05 products, fp32 accumulate)",
         "tf32x3": "f32 (tf32 hi/lo split operands, 3 tcgen05 products, fp32 accumulate)",
         "tf32": "tf32", "bf16": "bf16", "fp32": "f32"}
TOLERANCE = {"strict": 1e-4, "tf32x3": 1e-4, "fp32": 1e-4, "bf16": 1e-2, "tf32": None}


def gpu_arm(args) -> None:
    import torch
    import torch.distributed as dist
    import demucs_b200 as D
    from demucs_b200 import perf

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    shard = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        from demucs_b200.distributed import Shard
        # the stems leave each GPU for the host from the rank that made them: nothing is replicated over NVLink
        shard = Shard(gather="none")

    label, length, shifts, _ = WORKLOADS[args.config]
    model, oracle_models, bag_weights = build_workload(args.config, args.mode, dev)
    eng = (model.models[0] if hasattr(model, "models") else model).engine()
    engines = [m.engine() for m in model.models] if hasattr(model, "models") else [eng]
    nseg = -(-length // STRIDE)          # configs[2]: 64 segments in all, 64/N per GPU (strong scaling)
    host_mix = synth_track(length).pin_memory()
    dev_mix = host_mix.to(dev)
    kw = dict(shifts=shifts, split=True, overlap=0.25, batch_size=args.batch, shard=shard)
    import random

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device():
        random.seed(0)
        return D.apply_model(model, dev_mix, device=dev, **kw)

    # End-to-end step = the public call a user makes, on HOST buffers: apply_model uploads the (pinned) mix, separates,
    # and hands back the stems in pinned host memory (each rank the samples it produced; over all ranks the reads
    # cover the result exactly once).  The copies are inside apply_model, hence inside the timed region.
    last = {}

    def step_e2e():
        random.seed(0)
        out = D.apply_model(model, host_mix, device=dev, **kw)
        a, b = shard.owned if shard is not None else (0, length)
        last["own"] = (a, b)
        return float(out[0, 0, 0, a]) if b > a else 0.0

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            result = None        # free the previous step's output before the next one allocates its own
            result = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms) / steps, result

    for _ in range(max(args.warmup, 3)):
        step_device()
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = sum(e.launches for e in engines)
    ms, stems = timed(step_device, args.steps)
    launches = torch.tensor([float(sum(e.launches for e in engines) - l0)], device=dev)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stems": stems})
    del stems
    for _ in range(2):
        step_e2e()
    ms_e2e, _ = timed(step_e2e, args.steps)
    from demucs_b200 import apply as _apply
    io = torch.tensor([float(_apply.LAST_IO["h2d_bytes"]), float(_apply.LAST_IO["d2h_bytes"])], dtype=torch.float64,
                      device=dev)      # counted by apply_model from the tensors it copied
    if world > 1:
        dist.all_reduce(io)
        dist.all_reduce(launches)
    track_s = length / SR
    units = workload_config(world, args.mode, args.batch, args.config)["segments"]     # segment forwards per step
    value, e2e = track_s / (ms / 1e3), track_s / (ms_e2e / 1e3)

    # weak-scaling companion (N > 1): 64 segments PER GPU, device-resident, same call
    weak = None
    if world > 1 and not args.no_weak and args.config == "configs2":
        wlen = SEGMENTS * world * STRIDE
        wmix = synth_track(wlen).to(dev)

        def step_weak():
            return D.apply_model(model, wmix, device=dev, **kw)
        step_weak()
        ms_w, _ = timed(step_weak, max(1, args.steps // 2))
        weak = {"value": (wlen / SR) / (ms_w / 1e3), "unit": UNIT, "ms_per_step": ms_w, "segments_per_gpu": SEGMENTS,
                "scaling": "weak"}
        del wmix

    # per-kernel device time + algorithmic work of ONE more step, with events around every launch
    prof = perf.profile_step(eng, step_device)
    # spot-check window (big configs): EVERY rank takes part in the sharded call -- it is a collective -- and rank 0,
    # whose samples the window lies in, keeps the slice for the comparison with the oracle further down
    window = (2 * STRIDE + 100000, 2 * STRIDE + 120000)
    got_window = None
    if args.config != "configs2" and not args.no_cpu:
        random.seed(0)
        got_window = D.apply_model(model, dev_mix, device=dev, **kw)[..., window[0]:window[1]].cpu()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peaks = measured_peaks()
    top = prof["dominant"]
    # tensor-pipe peak the dominant kernel's MMAs run against: kind::f16 (bf16) for the bf16-operand modes, half of it
    # for kind::tf32.  `achieved` counts ALGORITHMIC flops (2*M*N*K); the split-operand modes issue three MMAs per product.
    # ("bf16" mode: only the transformer's kernels -- 64-element k-blocks, attention -- issue bf16 MMAs; its U-Net
    # convolutions are single-pass tf32)
    b16 = args.mode == "strict" or (args.mode == "bf16" and (top["name"].startswith("conv_gemm_tc<64") or
                                                             top["name"].startswith("attention")))
    tensor_peak = peaks["bf16_tflops"] if b16 else peaks["bf16_tflops"] / 2.0
    passes = 3 if args.mode in ("strict", "tf32x3") else 1
    if top["bound"] == "tensor":
        achieved, peak, unit = top["tflops"], tensor_peak, "TFLOP/s"
    else:
        achieved, peak, unit = top["gbs"], peaks["hbm_gbs"], "GB/s"
    ncu = ncu_traffic(top["name"], args.mode)
    if ncu:   # the ncu pass ran 16-segment forwards; activations (all but the L2-resident weights) scale with the batch
        ncu["captured_at_batch"] = 16
        ncu["bytes_per_launch"] *= min(args.batch, nseg // world) / 16
    roofline = {"kernel": top["name"], "bound": top["bound"], "achieved": achieved, "peak": peak, "unit": unit,
                "frac": achieved / peak, "traffic": ncu["bytes_per_launch"] if ncu else None,
                "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)", "ncu": ncu,
                "mma_passes_per_product": passes,
                "tensor_pipe_frac_incl_passes": (passes * achieved / peak) if top["bound"] == "tensor" else None,
                "algorithmic_bytes_per_launch": top.get("bytes_per_launch"), "peak_source": peaks["source"],
                "share_of_step": top["share"], "launches_per_step": top["count"],
                "avg_launch_ms": top["ms"] / max(top["count"], 1),
                "kernels": prof["table"]}
    cpu_baseline, parity = None, None
    if args.config != "configs2" and not args.no_cpu:
        # spot check on a sub-window of rank 0's samples: the oracle evaluates only the segments that touch it
        from oracle.apply_oracle import apply_model_oracle
        torch.set_num_threads(os.cpu_count() or 1)
        random.seed(0)
        with torch.no_grad():
            want = apply_model_oracle(oracle_models, host_mix, shifts=shifts, split=True, overlap=0.25,
                                      bag_weights=bag_weights, window=window)[..., window[0]:window[1]]
        got = got_window
        err = max(float((got[0, s_] - want[0, s_]).norm() / want[0, s_].norm()) for s_ in range(got.shape[1]))
        parity = {"against": "port (oracle, windowed)", "clip": f"output samples [{window[0]}, {window[1]}) of the track",
                  "mode": args.mode, "per_stem_rel_l2_max": err, "tolerance": TOLERANCE[args.mode],
                  "within_tolerance": (err <= TOLERANCE[args.mode]) if TOLERANCE[args.mode] else None}
    if world == 1 and not args.no_cpu and args.config == "configs2":
        threads = os.cpu_count() or 1
        nsamp = CPU_SAMPLE_SEGMENTS
        times, kind, (cpu_mix, cpu_out) = cpu_apply_seconds(nsamp * STRIDE, 2, threads, want_output=True)
        sec = times[-1]
        # the CPU run doubles as the checker: same weights, same samples, through the same public call
        got = D.apply_model(model, cpu_mix, shifts=0, split=True, overlap=0.25, device=dev, batch_size=args.batch)
        err = max(float((got[0, s] - cpu_out[0, s]).norm() / cpu_out[0, s].norm()) for s in range(got.shape[1]))
        parity = {"against": kind, "clip": f"first {nsamp} segments of the bench track, shifts=0, overlap=0.25",
                  "mode": args.mode, "per_stem_rel_l2_max": err, "tolerance": TOLERANCE[args.mode],
                  "within_tolerance": (err <= TOLERANCE[args.mode]) if TOLERANCE[args.mode] else None}
        cpu_baseline = {"value": (nsamp * STRIDE / SR) / sec, "unit": UNIT, "cores": threads, "kind": kind,
                        "sample": f"second of 2 x apply_model on the first {nsamp} segments ({nsamp * STRIDE / SR:.1f} s) of "
                                  f"the bench track, {threads} threads, torch {torch.__version__} CPU fp32"}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak",
            "vs_baseline": None, "dtype": DTYPE[args.mode], "data": "synthetic",
            "config": workload_config(world, args.mode, args.batch, args.config),
            "e2e": {"value": e2e, "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(io[0]),
                    "d2h_bytes_per_step": int(io[1]),
                    "api": "demucs_b200.apply_model(model, pinned host mix) -> pinned host stems"},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
            "parity": parity, "weak": weak,
            "model_roofline": {"segments_per_s": units / (ms / 1e3),
                               "tf32_roofline_segments_per_s_per_gpu": 1e3 / 0.742,
                               "bf16_roofline_segments_per_s_per_gpu": 1e3 / 0.377,
                               "frac_of_tf32_model_roofline": (units / world / (ms / 1e3)) / (1e3 / 0.742)}}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def hdemucs_arm(args) -> None:
    """BASELINE configs[1]: the hdemucs_mmi architecture (Hybrid Demucs v3, 83.6 M parameters, no transformer), forward of
    a batch of 16 x 7.8 s segments on one B200.  value: audio-seconds per second with the batch resident in HBM; e2e: the
    same from pinned host memory and back; parity: one item against the CPU oracle."""
    import torch
    from demucs_b200 import hdemucs as HD, perf
    from demucs_b200.hdemucs_engine import HDemucsEngine
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    cfg = HD.hdemucs_mmi_config()
    W = HD.init_weights(cfg, 0)
    mode = args.mode or "strict"
    eng = HDemucsEngine(cfg, W, dev, mode=mode)
    B, L = 16, SEG_LEN
    host = (0.1 * torch.randn(B, 2, L, generator=torch.Generator().manual_seed(1234))).pin_memory()
    x = host.to(dev)
    out = torch.empty(B, 4, 2, L, device=dev)
    host_out = torch.empty(B, 4, 2, L).pin_memory()

    def step():
        eng.forward(x, out=out)

    def step_e2e():
        xd = host.to(dev, non_blocking=True)
        eng.forward(xd, out=out)
        host_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, steps):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    for _ in range(max(args.warmup, 3)):
        step()
    sampler = ClockSampler(0)
    l0 = eng.launches
    ms = timed(step, args.steps)
    launches = eng.launches - l0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"stems": out})
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    prof = perf.profile_step(eng, step)
    peaks = measured_peaks()
    top = prof["dominant"]
    if top["bound"] == "tensor":
        achieved, peak, unit = top["tflops"], peaks["bf16_tflops"], "TFLOP/s"
    else:
        achieved, peak, unit = top["gbs"], peaks["hbm_gbs"], "GB/s"
    parity = cpu_baseline = None
    if not args.no_cpu:
        from oracle.hdemucs_oracle import hdemucs_forward
        torch.set_num_threads(os.cpu_count() or 1)
        with torch.no_grad():
            hdemucs_forward(W, cfg, host[:1])
            t0 = time.perf_counter()
            want = hdemucs_forward(W, cfg, host[:2])
            sec = time.perf_counter() - t0
        got = eng.forward(x[:2].contiguous()).cpu()
        err = max(float((got[:, s_] - want[:, s_]).norm() / want[:, s_].norm()) for s_ in range(4))
        parity = {"against": "port (oracle)", "clip": "items 0-1 of the batch", "mode": mode, "per_stem_rel_l2_max": err,
                  "tolerance": TOLERANCE[mode], "within_tolerance": err <= TOLERANCE[mode] if TOLERANCE[mode] else None}
        cpu_baseline = {"value": 2 * L / SR / sec, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                        "sample": f"one forward of 2 x 7.8 s items after a warm-up, torch {torch.__version__} CPU fp32"}
    audio_s = B * L / SR
    line = {"metric": "hdemucs_mmi audio-seconds separated per second (forward of 16 x 7.8 s)", "value": audio_s / (ms / 1e3),
            "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE[mode], "data": "synthetic",
            "config": {"workload": "hdemucs_mmi architecture (Hybrid Demucs v3, random-init, 83.6 M parameters): STFT + dual U-Net "
                                   "forward, batch 16 x 7.8 s segments on 1 B200 (BASELINE configs[1])", "name": "hdemucs_mmi",
                       "mode": mode, "l2": "activations of a step exceed L2 many times over"},
            "e2e": {"value": audio_s / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e, "h2d_bytes_per_step": host.numel() * 4,
                    "d2h_bytes_per_step": host_out.numel() * 4, "api": "HDemucsEngine.forward on a pinned host batch"},
            "gpu_launches": launches, "clocks": clocks,
            "roofline": {"kernel": top["name"], "bound": top["bound"], "achieved": achieved, "peak": peak, "unit": unit,
                         "frac": achieved / peak, "traffic": None, "share_of_step": top["share"], "kernels": prof["table"]},
            "cpu_baseline": cpu_baseline, "parity": parity}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="configs2", choices=list(WORKLOADS) + ["hdemucs_mmi"],
                    help="configs2 (default, the headline): 64 x 7.8 s segments; 6s_10min / ft_10min: BASELINE configs[3] / [4]")
    ap.add_argument("--mode", default=os.environ.get("BD_MODE"), choices=["fp32", "tf32", "tf32x3", "strict", "bf16"],
                    help="strict (default): error-compensated tensor-core arithmetic, per-stem rel-L2 <= 1e-4; "
                         "bf16: reduced precision, <= 1e-2")
    ap.add_argument("--batch", type=int, default=64, help="segments per forward (64: one forward per step and GPU, ~36 GB)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity leg")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling companion run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the stems of the last one as DIR/stems.npy (float32; beyond "
                         f"{DUMP_BYTES >> 20} MB, fixed seeded windows of {DUMP_WINDOW} samples along time); "
                         "the GPU arms need --gpus 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.gpus != 1 and args.impl != "reference":
        ap.error("--dump-outputs needs --gpus 1 (with more, each rank holds only the samples it produced)")
    if args.config == "hdemucs_mmi" and args.impl != "reference":
        return hdemucs_arm(args)
    if args.mode is None:
        args.mode = WORKLOADS.get(args.config, WORKLOADS["configs2"])[3]
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
