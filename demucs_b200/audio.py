"""Audio front and back door on the device -- drop-in for the tensor side of reference ``demucs/audio.py``.

``convert_audio_channels`` / ``convert_audio`` (audio.py:143-172), ``prevent_clip`` (audio.py:218-233), ``i16_pcm``
(audio.py:175-180) and ``save_audio`` (audio.py:236-265) with the reference's names, arguments and error behaviour, for
CUDA tensors: channel conversion and ``julius.resample_frac`` as one polyphase kernel, clip prevention + PCM
quantisation + interleaving as one kernel, so that a stem crosses PCIe as 16-bit frames.  There is no CPU path:
CPU tensors raise ``KernelError`` (use the reference, or move the tensor to the GPU).

``julius`` is a third-party dependency that is not vendored in the reference tree (requirements.txt: julius>=0.2.3)
and not installed here; the filter bank below restates its published algorithm (julius/resample.py, ResampleFrac:
zeros=24, rolloff=0.945, Hann-windowed sinc, every phase normalised to unit sum, replicate padding, floor output
length) -- parity with julius itself is UNPINNED, see oracle/audio_oracle.py.  ``save_audio`` writes RIFF/WAVE itself,
and ``load_audio`` reads it: the header is parsed on the host, the data chunk goes to the GPU in its own encoding and one
kernel decodes, de-interleaves and converts its channels.  Other containers (mp3, flac, ...) and mp3 / flac encoding
stay outside.
"""
from __future__ import annotations

import math
import os
import struct
import typing as tp
from pathlib import Path

import torch

from . import _lib
from ._lib import ptr

_CLIP = {None: 0, "none": 0, "rescale": 1, "clamp": 2, "tanh": 3}
_KERNELS: tp.Dict[tp.Tuple, tp.Tuple[torch.Tensor, int, int, int]] = {}


def _require_cuda(wav: torch.Tensor, what: str) -> None:
    if wav.device.type != "cuda" and _lib.TEST_HOOK is None:
        raise _lib.KernelError(f"demucs_b200.audio.{what} runs on CUDA tensors only (there is no CPU path)")


def _stream(wav: torch.Tensor) -> int:
    return torch.cuda.current_stream(wav.device).cuda_stream if wav.device.type == "cuda" else 0


def resample_kernel(old_sr: int, new_sr: int, zeros: int = 24, rolloff: float = 0.945):
    """julius.ResampleFrac._init_kernels: ([new_sr, 2*width + old_sr] float32 filter bank, old_sr, new_sr, width), the
    rates reduced by their gcd."""
    gcd = math.gcd(old_sr, new_sr)
    old_sr, new_sr = old_sr // gcd, new_sr // gcd
    sr = min(new_sr, old_sr) * rolloff
    width = math.ceil(zeros * old_sr / sr)
    idx = torch.arange(-width, width + old_sr).float()
    kernels = []
    for i in range(new_sr):
        t = (-i / new_sr + idx / old_sr) * sr
        t = t.clamp_(-zeros, zeros)
        t *= math.pi
        window = torch.cos(t / zeros / 2) ** 2
        kernel = torch.where(t == 0, torch.ones_like(t), torch.sin(t) / t) * window
        kernel.div_(kernel.sum())
        kernels.append(kernel)
    return torch.stack(kernels).contiguous(), old_sr, new_sr, width


def convert_audio_channels(wav: torch.Tensor, channels: int = 2) -> torch.Tensor:
    """audio.py:143-166 for a CUDA tensor [..., src_channels, length]."""
    *shape, src_channels, length = wav.shape
    if src_channels == channels:
        return wav
    if not (channels == 1 or src_channels == 1 or src_channels >= channels):
        raise ValueError('The audio file has less channels than requested but is not mono.')
    _require_cuda(wav, "convert_audio_channels")
    x = wav.contiguous().float()
    items = int(math.prod(shape)) if shape else 1
    y = torch.empty(*shape, channels, length, dtype=torch.float32, device=wav.device)
    with torch.cuda.device(wav.device) if wav.device.type == "cuda" else _null():
        _lib.call("bd_convert_channels", ptr(x), ptr(y), items, src_channels, channels, length, _stream(wav))
    return y


def convert_audio(wav: torch.Tensor, from_samplerate: int, to_samplerate: int, channels: int) -> torch.Tensor:
    """audio.py:169-172: to ``channels`` channels, then ``julius.resample_frac(wav, from_samplerate, to_samplerate)``
    (output length floor(length * to / from)) -- one kernel for both."""
    *shape, src_channels, length = wav.shape
    if from_samplerate == to_samplerate:
        return convert_audio_channels(wav, channels)
    if not (src_channels == channels or channels == 1 or src_channels == 1 or src_channels >= channels):
        raise ValueError('The audio file has less channels than requested but is not mono.')
    _require_cuda(wav, "convert_audio")
    key = (int(from_samplerate), int(to_samplerate), str(wav.device))
    if key not in _KERNELS:
        k, o, n, w = resample_kernel(int(from_samplerate), int(to_samplerate))
        _KERNELS[key] = (k.to(wav.device), o, n, w)
    kern, old_sr, new_sr, width = _KERNELS[key]
    out_len = int(new_sr * length // old_sr)
    x = wav.contiguous().float()
    items = int(math.prod(shape)) if shape else 1
    y = torch.empty(*shape, channels, out_len, dtype=torch.float32, device=wav.device)
    if out_len:
        with torch.cuda.device(wav.device) if wav.device.type == "cuda" else _null():
            _lib.call("bd_resample_frac", ptr(x), ptr(y), ptr(kern), items, src_channels, channels, length, out_len, old_sr,
                      new_sr, width, _stream(wav))
    return y


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def _clip_pcm(wav: torch.Tensor, clip, bits: int) -> torch.Tensor:
    """wav [channels, frames] (CUDA float) -> [frames, channels] int16 / int32(24-bit) / float32, clip prevention applied."""
    if clip not in _CLIP:
        raise ValueError(f"Invalid mode {clip}")
    if not wav.dtype.is_floating_point:
        raise AssertionError("too late for clipping")
    _require_cuda(wav, "prevent_clip / PCM")
    if wav.dim() != 2:
        raise ValueError("expected wav of shape [channels, frames]")
    x = wav.contiguous().float()
    C_, T = x.shape
    out = torch.empty(T, C_, dtype={16: torch.int16, 24: torch.int32, 32: torch.float32}[bits], device=wav.device)
    peak = torch.empty(1, dtype=torch.float32, device=wav.device)
    with torch.cuda.device(wav.device) if wav.device.type == "cuda" else _null():
        if _CLIP[clip] == 1:
            _lib.call("bd_absmax", ptr(x), ptr(peak), x.numel(), _stream(wav))
        if T:
            _lib.call("bd_clip_pcm", ptr(x), ptr(out), C_, T, _CLIP[clip], ptr(peak), bits, _stream(wav))
    return out


def prevent_clip(wav: torch.Tensor, mode: tp.Optional[str] = 'rescale') -> torch.Tensor:
    """audio.py:218-233 (``wav`` [channels, frames] or [..., frames]; returns the same layout)."""
    if mode is None or mode == 'none':
        return wav
    assert wav.dtype.is_floating_point, "too late for clipping"
    if mode not in _CLIP:
        raise ValueError(f"Invalid mode {mode}")
    flat = wav.reshape(1, -1)
    return _clip_pcm(flat, mode, 32).reshape(-1).view(wav.shape)      # one channel: interleaving is the identity


def i16_pcm(wav: torch.Tensor) -> torch.Tensor:
    """audio.py:175-180: float -> int16 (clamp to [-1, 1], * 32767, truncate); integer input is returned as is."""
    if not wav.dtype.is_floating_point:
        return wav
    return _clip_pcm(wav.reshape(1, -1), "none", 16).reshape(-1).view(wav.shape)


def stems_to_pcm(wav: torch.Tensor, clip: tp.Optional[str] = 'rescale', bits_per_sample: int = 16,
                 as_float: bool = False) -> torch.Tensor:
    """The back door: wav [channels, frames] on the GPU -> interleaved frames [frames, channels] on the HOST (pinned),
    clip prevention and quantisation done on the device, so 2 (or 4) bytes per sample cross PCIe."""
    bits = 32 if as_float else int(bits_per_sample)
    if bits == 32 and not as_float:
        raise ValueError("32-bit integer PCM is not produced; use as_float=True for 32-bit float")
    dev = _clip_pcm(wav, clip, bits)
    host = torch.empty(dev.shape, dtype=dev.dtype, pin_memory=dev.device.type == "cuda")
    host.copy_(dev, non_blocking=True)
    if dev.device.type == "cuda":
        torch.cuda.current_stream(dev.device).synchronize()
    return host


def save_audio(wav: torch.Tensor, path: tp.Union[str, Path], samplerate: int, bitrate: int = 320,
               clip: tp.Optional[str] = 'rescale', bits_per_sample: int = 16, as_float: bool = False, preset: int = 2):
    """audio.py:236-265 for ``.wav`` targets: clip prevention, quantisation and interleaving on the device, then a
    RIFF/WAVE file written directly (PCM_S 16 / 24 bit or IEEE float 32).  mp3 / flac need lameenc / torchaudio, which
    are outside this build."""
    path = Path(path)
    suffix = path.suffix.lower()
    if suffix in (".mp3", ".flac"):
        raise ValueError(f"{suffix} encoding is outside this build (lameenc / torchaudio); write .wav")
    if suffix != ".wav":
        raise ValueError(f"Invalid suffix for path: {suffix}")
    frames = stems_to_pcm(wav, clip, bits_per_sample, as_float)
    bits = 32 if as_float else int(bits_per_sample)
    n, ch = frames.shape
    if bits == 24:      # int32 container -> packed little-endian 3-byte samples
        data = frames.numpy().astype("<i4").view("u1").reshape(n, ch, 4)[..., :3].tobytes()
    else:
        data = frames.numpy().tobytes()
    block = ch * bits // 8
    fmt = 3 if as_float else 1
    header = b"RIFF" + struct.pack("<I", 36 + len(data)) + b"WAVE" + b"fmt " + struct.pack(
        "<IHHIIHH", 16, fmt, ch, samplerate, samplerate * block, block, bits) + b"data" + struct.pack("<I", len(data))
    with open(path, "wb") as f:
        f.write(header)
        f.write(data)


_PCM = {(1, 8): 1, (1, 16): 2, (1, 24): 3, (1, 32): 4, (3, 32): 5, (3, 64): 6}     # (format tag, bits) -> BD_PCM_*
_TAG_NAMES = {2: "MS ADPCM", 6: "A-law", 7: "\u00b5-law", 0x11: "IMA ADPCM"}
_CONTAINERS = {b"RIFX": "RIFX (big-endian RIFF)", b"RF64": "RF64", b"BW64": "BW64", b"riff": "Sony Wave64"}
_GUID_TAIL = bytes.fromhex("000000001000800000aa00389b71")      # KSDATAFORMAT_SUBTYPE_* after the 2-byte format tag
# Bytes of one pinned staging buffer (rounded down to whole frames) and how many of them are in flight: pinned memory
# stays bounded whatever the file's size, and the file read of one chunk overlaps the copy and decode of the previous.
_CHUNK_BYTES = 4 << 20
_RING = 3


class _WavData(tp.NamedTuple):
    pcm: int            # BD_PCM_*
    channels: int
    samplerate: int
    block: int          # bytes per frame
    offset: int         # file offset of the first frame
    frames: int


def _wav_fmt(body: bytes) -> tp.Tuple[int, int, int, int]:
    """The ``fmt `` chunk -> (BD_PCM_*, channels, sample rate, bytes per frame)."""
    if len(body) < 16:
        raise ValueError(f"fmt chunk of {len(body)} bytes (at least 16 expected)")
    tag, channels, samplerate, _, _, bits = struct.unpack("<HHIIHH", body[:16])
    if tag == 0xFFFE:           # WAVE_FORMAT_EXTENSIBLE: the real tag heads the sub-format GUID; wValidBitsPerSample is
        if len(body) < 40:      # ignored, samples are scaled by their container size (as ffmpeg does)
            raise ValueError(f"WAVE_FORMAT_EXTENSIBLE fmt chunk of {len(body)} bytes (40 expected)")
        if body[26:40] != _GUID_TAIL:
            raise ValueError("WAVE_FORMAT_EXTENSIBLE with a sub-format GUID that is not a WAVE format tag")
        tag = struct.unpack("<H", body[24:26])[0]
    if tag not in (1, 3):
        name = _TAG_NAMES.get(tag, "unsupported")
        raise ValueError(f"WAVE format tag 0x{tag:04x} ({name}) is not decoded: PCM and IEEE float only")
    if channels == 0:
        raise ValueError("the fmt chunk declares zero channels")
    if (tag, bits) not in _PCM:
        kind = "integer PCM: 8, 16, 24 or 32" if tag == 1 else "IEEE float: 32 or 64"
        raise ValueError(f"{bits} bits per sample is not decoded ({kind} bits)")
    if samplerate == 0:
        raise ValueError("the fmt chunk declares a sample rate of 0")
    return _PCM[(tag, bits)], channels, samplerate, channels * bits // 8


def _wav_layout(f: tp.BinaryIO, size: int) -> _WavData:
    """Walks the RIFF chunks up to ``data``: chunks of other ids are skipped with their pad byte; a data size of 0,
    0xFFFFFFFF or past the end of the file (streaming encoders) means the bytes present; a partial last frame is
    dropped."""
    head = f.read(12)
    if head[:4] in _CONTAINERS:
        raise ValueError(f"{_CONTAINERS[head[:4]]} files are not decoded: little-endian RIFF/WAVE only")
    if len(head) < 12 or head[:4] != b"RIFF" or head[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE file")
    fmt = None
    pos = 12
    while True:
        f.seek(pos)
        ck = f.read(8)
        if len(ck) < 8:
            break
        cid, n = ck[:4], struct.unpack("<I", ck[4:])[0]
        if cid == b"fmt ":
            fmt = _wav_fmt(f.read(n))
        elif cid == b"data":
            if fmt is None:
                break
            pcm, channels, samplerate, block = fmt
            avail = size - (pos + 8)
            frames = (n if 0 < n <= avail else avail) // block
            if frames == 0:
                raise ValueError("the data chunk holds no complete frame")
            return _WavData(pcm, channels, samplerate, block, pos + 8, frames)
        pos += 8 + n + (n & 1)
    raise ValueError("no fmt chunk before the data chunk" if fmt is None else "no data chunk")


def _read_into(f: tp.BinaryIO, buf: memoryview) -> None:
    got = 0
    while got < len(buf):
        n = f.readinto(buf[got:])
        if not n:
            raise ValueError("the file ended inside its data chunk")
        got += n


def load_audio(path: tp.Union[str, Path], samplerate: tp.Optional[int] = None, channels: tp.Optional[int] = None,
               device: tp.Union[str, torch.device] = "cuda") -> tp.Tuple[torch.Tensor, int]:
    """A RIFF/WAVE file -> (wav [channels, length] float32 on ``device``, its sample rate).

    Integer PCM (8 bit unsigned, 16 / 24 / 32 bit signed) and IEEE float (32 / 64 bit), plain or
    WAVE_FORMAT_EXTENSIBLE, scaled to [-1, 1) as ``torchaudio.load(normalize=True)`` and ffmpeg do.  The data chunk
    crosses PCIe in its own encoding (a 16-bit file at half the bytes of float) through a small ring of pinned buffers,
    and ``bd_pcm_decode`` de-interleaves and scales it on the device.  ``channels``: convert as
    ``convert_audio_channels`` does, in the same kernel.  ``samplerate``: resample with ``convert_audio`` (and return
    that rate).  Other containers and codecs (RF64, A-law, ADPCM, ...) raise ``ValueError`` naming the reason."""
    device = torch.device(device)
    with open(path, "rb") as f:
        info = _wav_layout(f, os.fstat(f.fileno()).st_size)
        dst_ch = info.channels if channels is None else int(channels)
        if dst_ch < 1 or not (dst_ch == info.channels or dst_ch == 1 or info.channels == 1 or info.channels >= dst_ch):
            raise ValueError('The audio file has less channels than requested but is not mono.')
        wav = torch.empty(dst_ch, info.frames, dtype=torch.float32, device=device)
        _require_cuda(wav, "load_audio")
        on_cuda = device.type == "cuda"
        total = info.frames * info.block
        chunk = min(max(_CHUNK_BYTES // info.block, 1) * info.block, total)
        host = [torch.empty(chunk, dtype=torch.uint8, pin_memory=on_cuda) for _ in range(min(_RING, -(-total // chunk)))]
        copied: tp.List[tp.Optional[torch.cuda.Event]] = [None] * len(host)
        staged = torch.empty(chunk, dtype=torch.uint8, device=device)   # copy i + 1 follows decode i on the stream
        f.seek(info.offset)
        with torch.cuda.device(device) if on_cuda else _null():
            for i, off in enumerate(range(0, total, chunk)):
                slot = i % len(host)
                if copied[slot] is not None:
                    copied[slot].synchronize()          # the copy that last read this buffer has finished
                n = min(chunk, total - off)
                _read_into(f, memoryview(host[slot].numpy())[:n])
                staged[:n].copy_(host[slot][:n], non_blocking=on_cuda)
                if on_cuda:
                    copied[slot] = torch.cuda.current_stream(device).record_event()
                _lib.call("bd_pcm_decode", ptr(staged), ptr(wav), info.pcm, info.channels, dst_ch, n // info.block,
                          info.frames, off // info.block, _stream(wav))
    if samplerate is not None and samplerate != info.samplerate:
        return convert_audio(wav, info.samplerate, samplerate, dst_ch), samplerate
    return wav, info.samplerate
