"""WAV input on the device: path-to-device time of ``demucs_b200.audio.load_audio`` for a 10-minute 44.1 kHz stereo
file (s16, s24, f32), the ``bd_pcm_decode`` kernel rate (CUDA events), and numpy decode + a float32 host->device copy
of the same file for comparison.

    python tools/wav_load_bench.py [--out DIR] [--seconds 600] [--reps 5]

The files are written from a seeded signal into DIR (default: a temporary directory, removed afterwards) and each is
read once before its timed reads, so every timed read comes from the page cache: the numbers are the host and PCIe
side of loading, not the disk.  The decode kernel's working set (encoded + decoded bytes, 318 MB for s16) exceeds the
126 MB L2.  Prints one JSON line per format, then one with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from demucs_b200 import _lib, audio as A  # noqa: E402

HBM_DATASHEET_GBS = 7700.0          # HGX B200 data sheet, per GPU; a bound, not a measured rate
DEV = "cuda:0"
HEADER = 44                         # save_audio writes the canonical 44-byte header
FORMATS = {"s16": (dict(bits_per_sample=16), 2), "s24": (dict(bits_per_sample=24), 3), "f32": (dict(as_float=True), 5)}


def card() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as err:
        q = f"unavailable: {err}"
    return {"card": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": q}


def numpy_load(path: str, kind: str) -> torch.Tensor:
    """The host alternative: decode with numpy, then copy float32 planes to the device (pageable)."""
    raw = np.fromfile(path, dtype=np.uint8, offset=HEADER)
    if kind == "s16":
        x = raw.view("<i2").astype(np.float32) / np.float32(2 ** 15)
    elif kind == "s24":
        t = raw.reshape(-1, 3).astype(np.int32)
        v = ((t[:, 0] | (t[:, 1] << 8) | (t[:, 2] << 16)) << 8) >> 8
        x = v.astype(np.float32) / np.float32(2 ** 23)
    else:
        x = raw.view("<f4")
    return torch.from_numpy(np.ascontiguousarray(x.reshape(-1, 2).T)).to(DEV)


def host_timed(fn, reps: int):
    fn()                                  # warm-up: page cache, pinned staging buffers, module load
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    return out, times


def kernel_rate(path: str, pcm: int, frames: int, launches: int = 20) -> dict:
    enc = torch.from_numpy(np.fromfile(path, dtype=np.uint8, offset=HEADER)).to(DEV)
    out = torch.empty(2, frames, device=DEV)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        _lib.call("bd_pcm_decode", enc.data_ptr(), out.data_ptr(), pcm, 2, 2, frames, frames, 0, stream)

    for _ in range(3):
        launch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(launches):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / launches
    nbytes = enc.numel() + out.numel() * 4
    gbs = nbytes / ms / 1e6
    return {"kernel_ms": round(ms, 4), "kernel_bytes": nbytes, "kernel_gbs": round(gbs, 1),
            "kernel_frac_of_hbm_datasheet": round(gbs / HBM_DATASHEET_GBS, 3)}


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="directory for the generated WAV files (default: a temporary one)")
    ap.add_argument("--seconds", type=int, default=600)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wav_load_bench measures on a CUDA device; none is visible")
    _lib.build()
    sr = 44100
    tmp = None
    out_dir = args.out
    if out_dir is None:
        tmp = tempfile.TemporaryDirectory()
        out_dir = tmp.name
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)
    signal = torch.from_numpy(0.25 * rng.standard_normal((2, args.seconds * sr), dtype=np.float32)).to(DEV)
    try:
        for kind, (kw, pcm) in FORMATS.items():
            path = os.path.join(out_dir, f"wav_load_bench_{kind}.wav")
            A.save_audio(signal, path, sr, clip="none", **kw)
            size = os.path.getsize(path)
            wav, t_dev = host_timed(lambda: A.load_audio(path, device=DEV)[0], args.reps)
            ref, t_np = host_timed(lambda: numpy_load(path, kind), args.reps)
            res = {"format": kind, "seconds": args.seconds, "samplerate": sr, "channels": 2, "file_bytes": size,
                   "file_source": "page cache (read once before the timed reads)",
                   "load_audio_ms_median": round(1e3 * statistics.median(t_dev), 2),
                   "load_audio_ms_min": round(1e3 * min(t_dev), 2),
                   "numpy_then_h2d_ms_median": round(1e3 * statistics.median(t_np), 2),
                   "numpy_then_h2d_ms_min": round(1e3 * min(t_np), 2),
                   "speedup_median": round(statistics.median(t_np) / statistics.median(t_dev), 2),
                   "same_result": bool(torch.equal(wav, ref))}
            res.update(kernel_rate(path, pcm, wav.shape[1]))
            print(json.dumps(res), flush=True)
            del wav, ref
            if tmp is not None:
                os.remove(path)
    finally:
        if tmp is not None:
            tmp.cleanup()
    print(json.dumps(card()), flush=True)


if __name__ == "__main__":
    main()
