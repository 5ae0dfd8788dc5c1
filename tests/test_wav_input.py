"""WAV input on the device (demucs_b200/audio.py load_audio, csrc/audio.cu bd_pcm_decode, Separator.separate_audio_file).

The oracle is a numpy byte decode of the data chunk (``np.frombuffer``, 3-byte sign extension for s24) scaled by the
documented convention of ``torchaudio.load(normalize=True)`` and ffmpeg's f32 output: u8 (x - 128) / 2^7, s16 / 2^15,
s24 / 2^23, s32 round-to-nearest-even float / 2^31, f32 as is, f64 rounded once to f32; then the channel rule of
``convert_audio_channels`` with the mono down-mix summed in channel order.  It is pinned to that convention and not to
torchaudio itself, which cannot load files on this project's torch / torchaudio 2.11 stack without torchcodec.

CPU: the host logic (RIFF parser, staging ring, chunk placement, Separator plumbing) with the oracle registered as
the emulated ``bd_pcm_decode``.  GPU: the kernel and the whole path against the oracle, bitwise.
"""
import ctypes as C
import struct
import sys
import types

import numpy as np
import pytest
import torch
from scipy.io import wavfile

import abi_emulator
from _fixtures import rel_l2
from abi_emulator import emulated_abi
from demucs_b200 import _lib
from demucs_b200 import audio as A

U8, S16, S24, S32, F32, F64 = 1, 2, 3, 4, 5, 6
BPS = {U8: 1, S16: 2, S24: 3, S32: 4, F32: 4, F64: 8}
TAG_BITS = {U8: (1, 8), S16: (1, 16), S24: (1, 24), S32: (1, 32), F32: (3, 32), F64: (3, 64)}
GUID_TAIL = bytes.fromhex("000000001000800000aa00389b71")


def decode_oracle(payload: bytes, pcm: int, channels: int) -> np.ndarray:
    """Data-chunk bytes -> [channels, frames] float32 (a partial last frame is dropped)."""
    bps = BPS[pcm]
    n = len(payload) // (bps * channels)
    b = np.frombuffer(payload, np.uint8, n * bps * channels)
    if pcm == U8:
        x = (b.astype(np.float32) - np.float32(128)) / np.float32(2 ** 7)
    elif pcm == S16:
        x = b.view("<i2").astype(np.float32) / np.float32(2 ** 15)
    elif pcm == S24:
        t = b.reshape(-1, 3).astype(np.int32)
        v = t[:, 0] | (t[:, 1] << 8) | (t[:, 2] << 16)
        x = np.where(v >= 1 << 23, v - (1 << 24), v).astype(np.float32) / np.float32(2 ** 23)
    elif pcm == S32:
        x = b.view("<i4").astype(np.float32) / np.float32(2 ** 31)
    elif pcm == F32:
        x = b.view("<f4").copy()
    else:
        x = b.view("<f8").astype(np.float32)
    return np.ascontiguousarray(x.reshape(n, channels).T)


def channel_rule(x: np.ndarray, dst) -> np.ndarray:
    src = x.shape[0]
    if dst is None or dst == src:
        return x
    if dst == 1:
        s = np.zeros(x.shape[1], np.float32)
        for k in range(src):
            s = s + x[k]
        return (s / np.float32(src))[None]
    if src == 1:
        return np.repeat(x, dst, axis=0)
    return x[:dst].copy()


def _emulated_pcm_decode(src, dst, pcm, src_ch, dst_ch, frames, dst_ld, frame0, stream):
    y = channel_rule(decode_oracle(C.string_at(src, frames * src_ch * BPS[pcm]), pcm, src_ch), dst_ch)
    abi_emulator.f32(dst, dst_ch * dst_ld).reshape(dst_ch, dst_ld)[:, frame0:frame0 + frames] = y


@pytest.fixture
def emu(monkeypatch):
    monkeypatch.setitem(abi_emulator.TABLE, "bd_pcm_decode", _emulated_pcm_decode)
    with emulated_abi():
        yield


def chunk(cid: bytes, body: bytes) -> bytes:
    return cid + struct.pack("<I", len(body)) + body + (b"\0" if len(body) % 2 else b"")


def fmt_body(pcm: int, channels: int, sr: int, extensible: bool = False, valid_bits=None, tag=None) -> bytes:
    ftag, bits = TAG_BITS[pcm]
    block = channels * bits // 8
    if not extensible:
        return struct.pack("<HHIIHH", ftag if tag is None else tag, channels, sr, sr * block, block, bits)
    sub = struct.pack("<H", ftag if tag is None else tag) + GUID_TAIL
    return struct.pack("<HHIIHH", 0xFFFE, channels, sr, sr * block, block, bits) + struct.pack(
        "<HHI", 22, valid_bits or bits, 0) + sub


def wav_file(path, payload: bytes, fmt: bytes, before=b"", after=b"", data_size=None, magic=b"RIFF"):
    data = b"data" + struct.pack("<I", len(payload) if data_size is None else data_size) + payload
    data += b"\0" if len(payload) % 2 and after else b""
    body = b"WAVE" + chunk(b"fmt ", fmt) + before + data + after
    path.write_bytes(magic + struct.pack("<I", len(body)) + body)
    return path


def random_payload(pcm: int, channels: int, frames: int, seed: int) -> bytes:
    rng = np.random.default_rng(seed)
    if pcm == F32:
        x = (rng.standard_normal((frames, channels)) * 0.5).astype("<f4").reshape(-1)
        x[:4] = np.array([0.0, -0.0, 1e-40, -3.5], "<f4")[:x.size]
        return x.tobytes()
    if pcm == F64:
        x = (rng.standard_normal((frames, channels)) * 0.5).astype("<f8").reshape(-1)
        x[:4] = np.array([0.0, -0.0, 1e-300, 1.0 + 2.0 ** -30], "<f8")[:x.size]
        return x.tobytes()
    return rng.integers(0, 256, frames * channels * BPS[pcm], dtype=np.uint8).tobytes()


SCIPY_DTYPES = {U8: np.uint8, S16: np.int16, S32: np.int32, F32: np.float32, F64: np.float64}


def scipy_data(pcm, channels, frames, seed):
    return np.frombuffer(random_payload(pcm, channels, frames, seed), SCIPY_DTYPES[pcm]).reshape(frames, channels)


# ---------------------------------------------------------------------------------------------------- CPU (emulator)

@pytest.mark.parametrize("pcm", [U8, S16, S32, F32, F64])
def test_scipy_files_decode_to_the_oracle(tmp_path, emu, pcm):
    for channels in (1, 2, 6):
        data = scipy_data(pcm, channels, 1001, pcm * 10 + channels)
        path = tmp_path / f"{pcm}_{channels}.wav"
        wavfile.write(path, 32000, data)
        want = decode_oracle(data.tobytes(), pcm, channels)
        for dst in (None, 1, 2, 6):
            if dst not in (None, 1, channels) and channels != 1 and channels < dst:
                continue
            wav, sr = A.load_audio(path, channels=dst, device="cpu")
            assert sr == 32000 and wav.dtype == torch.float32
            got = wav.numpy()
            expect = channel_rule(want, dst)
            assert got.shape == expect.shape and np.array_equal(got.view(np.int32), expect.view(np.int32)), (channels, dst)


def test_scipy_float_files_carry_fmt18_and_fact(tmp_path):
    path = tmp_path / "f.wav"
    wavfile.write(path, 44100, np.zeros((10, 2), np.float32))
    raw = path.read_bytes()
    assert struct.unpack("<I", raw[16:20])[0] == 18 and b"fact" in raw[:64]


def test_s24_written_by_save_audio(tmp_path, emu):
    x = 0.4 * torch.randn(2, 3001, generator=torch.Generator().manual_seed(3))
    path = tmp_path / "p24.wav"
    A.save_audio(x, path, 44100, clip="none", bits_per_sample=24)
    want = decode_oracle(path.read_bytes()[44:], S24, 2)
    wav, sr = A.load_audio(path, device="cpu")
    assert sr == 44100 and np.array_equal(wav.numpy(), want)
    assert (wav - x.clamp(-1, 1)).abs().max() <= 2.0 ** -22      # the writer clamps and truncates x * (2^23 - 1)


@pytest.mark.parametrize("pcm,valid", [(S24, 20), (F32, 32), (S16, 12)])
def test_extensible_headers(tmp_path, emu, pcm, valid):
    payload = random_payload(pcm, 2, 777, 5)
    path = wav_file(tmp_path / "e.wav", payload, fmt_body(pcm, 2, 48000, extensible=True, valid_bits=valid))
    wav, sr = A.load_audio(path, device="cpu")
    assert sr == 48000 and np.array_equal(wav.numpy(), decode_oracle(payload, pcm, 2))   # scaled by the container size


def test_odd_list_chunks_before_and_after_data(tmp_path, emu):
    payload = random_payload(U8, 1, 333, 6)                   # odd data size: padded before the trailing chunk
    lst = chunk(b"LIST", b"INFOISFT\x05\x00\x00\x00abcd\x00")  # odd size, pad byte follows
    path = wav_file(tmp_path / "l.wav", payload, fmt_body(U8, 1, 8000), before=lst + chunk(b"bext", b"x" * 7),
                    after=lst)
    wav, _ = A.load_audio(path, device="cpu")
    assert np.array_equal(wav.numpy(), decode_oracle(payload, U8, 1))


@pytest.mark.parametrize("data_size", [0xFFFFFFFF, 0, "past the end"])
def test_streaming_data_sizes_and_truncated_frame(tmp_path, emu, data_size):
    payload = random_payload(S16, 2, 500, 7)
    cut = payload + payload[:3]                               # a partial trailing frame
    size = 4 * 10 ** 6 if data_size == "past the end" else data_size
    path = wav_file(tmp_path / "s.wav", cut, fmt_body(S16, 2, 44100), data_size=size)
    wav, _ = A.load_audio(path, device="cpu")
    assert wav.shape == (2, 500) and np.array_equal(wav.numpy(), decode_oracle(payload, S16, 2))


def test_truncated_frame_with_an_honest_size(tmp_path, emu):
    payload = random_payload(S24, 6, 100, 8)
    path = wav_file(tmp_path / "t.wav", payload[:-5], fmt_body(S24, 6, 44100))
    wav, _ = A.load_audio(path, device="cpu")
    assert wav.shape == (6, 99) and np.array_equal(wav.numpy(), decode_oracle(payload, S24, 6)[:, :99])


@pytest.mark.parametrize("pcm,channels", [(S16, 2), (S24, 6), (F64, 1)])
def test_chunked_transfer_equals_one_chunk(tmp_path, monkeypatch, emu, pcm, channels):
    payload = random_payload(pcm, channels, 10000, 9)
    path = wav_file(tmp_path / "c.wav", payload, fmt_body(pcm, channels, 44100))
    whole, _ = A.load_audio(path, channels=1, device="cpu")
    block = BPS[pcm] * channels
    monkeypatch.setattr(A, "_CHUNK_BYTES", 7 * block + 3)     # 7 frames a chunk, the ring reused many times
    abi_emulator.CALLS.clear()
    pieces, _ = A.load_audio(path, channels=1, device="cpu")
    assert abi_emulator.CALLS.count("bd_pcm_decode") == -(-10000 // 7)
    assert np.array_equal(pieces.numpy(), whole.numpy())
    assert np.array_equal(whole.numpy(), channel_rule(decode_oracle(payload, pcm, channels), 1))


def test_load_audio_resamples_with_convert_audio(tmp_path, emu):
    payload = random_payload(S16, 1, 4800, 10)
    path = wav_file(tmp_path / "r.wav", payload, fmt_body(S16, 1, 48000))
    wav, sr = A.load_audio(path, 44100, 2, device="cpu")
    want = A.convert_audio(torch.from_numpy(decode_oracle(payload, S16, 1)), 48000, 44100, 2)
    assert sr == 44100 and torch.equal(wav, want)


def _rejects():
    pl = bytes(64)
    return {
        "RIFX": lambda p: wav_file(p, pl, fmt_body(S16, 2, 8000), magic=b"RIFX"),
        "RF64": lambda p: wav_file(p, pl, fmt_body(S16, 2, 8000), magic=b"RF64"),
        "Wave64": lambda p: p.write_bytes(b"riff\x2e\x91\xcf\x11\xa5\xd6\x28\xdb\x04\xc1\x00\x00" + bytes(64)),
        "A-law": lambda p: wav_file(p, pl, fmt_body(U8, 1, 8000, tag=6)),
        "µ-law": lambda p: wav_file(p, pl, fmt_body(U8, 1, 8000, tag=7)),
        "ADPCM": lambda p: wav_file(p, pl, fmt_body(S16, 1, 8000, tag=2)),
        "0x0055": lambda p: wav_file(p, pl, fmt_body(S16, 1, 8000, tag=0x55)),
        "IMA ADPCM": lambda p: wav_file(p, pl, fmt_body(S16, 1, 8000, extensible=True, tag=0x11)),
        "12 bits": lambda p: wav_file(p, pl, struct.pack("<HHIIHH", 1, 1, 8000, 16000, 2, 12)),
        "16 bits": lambda p: wav_file(p, pl, struct.pack("<HHIIHH", 3, 1, 8000, 16000, 2, 16)),
        "sub-format": lambda p: wav_file(p, pl, fmt_body(S16, 1, 8000, extensible=True)[:-1] + b"\x01"),
        "zero channels": lambda p: wav_file(p, pl, struct.pack("<HHIIHH", 1, 0, 8000, 0, 0, 16)),
        "no fmt chunk": lambda p: p.write_bytes(b"RIFF" + struct.pack("<I", 76) + b"WAVE" + chunk(b"data", pl)),
        "no data chunk": lambda p: p.write_bytes(b"RIFF" + struct.pack("<I", 28) + b"WAVE" + chunk(b"fmt ", fmt_body(S16, 1, 8000))),
        "no complete frame": lambda p: wav_file(p, b"\1\2\3", fmt_body(S16, 2, 8000)),
        "not a RIFF/WAVE": lambda p: p.write_bytes(b"fLaC" + bytes(60)),
    }


@pytest.mark.parametrize("reason", list(_rejects()))
def test_rejections_name_the_reason(tmp_path, emu, reason):
    path = tmp_path / "bad.wav"
    _rejects()[reason](path)
    with pytest.raises(ValueError, match=reason):
        A.load_audio(path, device="cpu")


def test_empty_data_chunk_is_rejected(tmp_path, emu):
    path = wav_file(tmp_path / "e.wav", b"", fmt_body(S16, 2, 8000))
    with pytest.raises(ValueError, match="no complete frame"):
        A.load_audio(path, device="cpu")


def test_channel_rule_and_device_are_checked(tmp_path):
    path = wav_file(tmp_path / "s.wav", random_payload(S16, 2, 10, 1), fmt_body(S16, 2, 8000))
    with emulated_abi(), pytest.raises(ValueError, match="less channels"):
        A.load_audio(path, channels=3, device="cpu")
    with pytest.raises(_lib.KernelError):                   # no CPU path outside the emulator
        A.load_audio(path, device="cpu")


def _v3_separator(D):
    from demucs_b200 import hdemucs as HD
    from oracle.make_golden import hdemucs_small_config
    cfg = hdemucs_small_config()
    cfg.segment = 2.0
    model = HD.HDemucs.from_config(cfg, init_seed=1, layer_scale=0.5, mode="fp32")
    return D.Separator(model, device="cpu", shifts=0)


def s24_payload(x: np.ndarray) -> bytes:
    """[channels, frames] float -> packed little-endian s24 frames"""
    v = np.clip(np.round(x.T * 2 ** 23), -2 ** 23, 2 ** 23 - 1).astype("<i4")
    return v.view(np.uint8).reshape(-1, 4)[:, :3].tobytes()


def test_separate_audio_file_host_logic(tmp_path, emu):
    """48 kHz mono s24 file on a v3 model under the emulated ABI: decoded, converted and separated exactly as
    separate_tensor separates the oracle's decode of the same bytes; host float32 results of the same shapes."""
    import demucs_b200 as D
    payload = s24_payload(0.3 * np.random.default_rng(8).standard_normal((1, 60000)))
    path = wav_file(tmp_path / "m.wav", payload, fmt_body(S24, 1, 48000))
    sep = _v3_separator(D)
    wav, stems = sep.separate_audio_file(path)
    want_wav, want = sep.separate_tensor(torch.from_numpy(decode_oracle(payload, S24, 1)), 48000)
    assert wav.device.type == "cpu" and wav.dtype == torch.float32 and torch.equal(wav, want_wav)
    assert list(stems) == list(want)
    for name, stem in stems.items():
        assert stem.device.type == "cpu" and stem.dtype == torch.float32 and stem.shape == want[name].shape
        assert torch.equal(stem, want[name]), name


def test_other_files_reach_torchaudio_and_errors_name_both_backends(tmp_path, monkeypatch, emu):
    import demucs_b200 as D
    from demucs_b200.api import LoadAudioError
    calls = []

    def failing_load(p):
        calls.append(p)
        raise RuntimeError("this torchaudio cannot decode it")

    fake = types.ModuleType("torchaudio")
    fake.load = failing_load
    monkeypatch.setitem(sys.modules, "torchaudio", fake)
    sep = _v3_separator(D)
    flac = tmp_path / "x.flac"
    flac.write_bytes(b"fLaC" + bytes(100))
    alaw = wav_file(tmp_path / "a.wav", bytes(64), fmt_body(U8, 1, 8000, tag=6))
    for path, reason in ((flac, "not a RIFF/WAVE file"), (alaw, "A-law")):
        with pytest.raises(LoadAudioError) as err:
            sep.separate_audio_file(path)
        msg = str(err.value)
        assert "using demucs_b200.audio.load_audio, got the following error" in msg and reason in msg
        assert "using torchaudio, got the following error: this torchaudio cannot decode it" in msg
        assert calls[-1] == str(path)
    fake.load = lambda p: (torch.full((2, 1000), 0.25), 44100)
    assert torch.equal(sep._load_audio(flac), torch.full((2, 1000), 0.25))       # torchaudio's result, as before


# ------------------------------------------------------------------------------------------------------------- GPU

DEV = "cuda:0"


@pytest.mark.gpu
@pytest.mark.parametrize("pcm", [U8, S16, S24, S32, F32, F64])
def test_gpu_kernel_matches_oracle(pcm):
    """Every format x (1, 2, 6 -> 1, 2) channels, frame counts that are no multiple of a CTA's tile, a source that
    does not start on a 16-byte boundary, and a frame0 / dst_ld window inside a larger output."""
    for src_ch in (1, 2, 6):
        for frames in (1, 4097, 70001):
            payload = random_payload(pcm, src_ch, frames, pcm * 100 + src_ch)
            for shift in (0, BPS[pcm] if BPS[pcm] != 3 else 1):
                buf = torch.zeros(len(payload) + 32, dtype=torch.uint8)
                buf[shift:shift + len(payload)] = torch.frombuffer(bytearray(payload), dtype=torch.uint8)
                src = buf.to(DEV)
                for dst_ch in (1, 2):
                    ld, frame0 = frames + 13, 5
                    out = torch.full((dst_ch, ld), float("nan"), device=DEV)
                    _lib.call("bd_pcm_decode", src.data_ptr() + shift, out.data_ptr(), pcm, src_ch, dst_ch, frames, ld,
                              frame0, torch.cuda.current_stream().cuda_stream)
                    got = out.cpu().numpy()
                    want = channel_rule(decode_oracle(payload, pcm, src_ch), dst_ch)
                    assert np.array_equal(got[:, frame0:frame0 + frames].view(np.int32), want.view(np.int32)), \
                        (pcm, src_ch, dst_ch, frames, shift)
                    assert np.isnan(got[:, :frame0]).all() and np.isnan(got[:, frame0 + frames:]).all()


@pytest.mark.gpu
def test_gpu_kernel_rejects_bad_arguments():
    src = torch.zeros(64, dtype=torch.uint8, device=DEV)
    out = torch.empty(2, 16, device=DEV)
    s = torch.cuda.current_stream().cuda_stream
    with pytest.raises(_lib.KernelError, match="aligned"):
        _lib.call("bd_pcm_decode", src.data_ptr() + 1, out.data_ptr(), S16, 2, 2, 8, 16, 0, s)
    with pytest.raises(_lib.KernelError, match="unknown format"):
        _lib.call("bd_pcm_decode", src.data_ptr(), out.data_ptr(), 7, 2, 2, 8, 16, 0, s)
    with pytest.raises(_lib.KernelError, match="less channels"):
        _lib.call("bd_pcm_decode", src.data_ptr(), out.data_ptr(), S16, 2, 3, 8, 16, 0, s)
    with pytest.raises(_lib.KernelError, match="bad sizes"):
        _lib.call("bd_pcm_decode", src.data_ptr(), out.data_ptr(), S16, 2, 2, 8, 10, 4, s)


@pytest.mark.gpu
def test_gpu_long_file_through_the_staging_ring(tmp_path):
    """60 s of stereo s16: more than two 4 MiB staging chunks, so every pinned buffer of the ring is reused."""
    frames = 60 * 44100
    assert frames * 4 > 2 * A._CHUNK_BYTES
    payload = random_payload(S16, 2, frames, 11)
    path = wav_file(tmp_path / "long.wav", payload, fmt_body(S16, 2, 44100), before=chunk(b"LIST", b"abc"))
    want = decode_oracle(payload, S16, 2)
    for dst in (None, 1):
        wav, sr = A.load_audio(path, channels=dst, device=DEV)
        assert wav.device.type == "cuda" and sr == 44100
        assert np.array_equal(wav.cpu().numpy(), channel_rule(want, dst))


@pytest.mark.gpu
@pytest.mark.parametrize("pcm,src_ch,dst_ch", [(S16, 1, 2), (S24, 6, 2), (F32, 2, 1), (F64, 2, 2)])
def test_gpu_load_audio_resamples_as_convert_audio(tmp_path, pcm, src_ch, dst_ch):
    payload = random_payload(pcm, src_ch, 48000 + 17, 12)
    path = wav_file(tmp_path / "r.wav", payload, fmt_body(pcm, src_ch, 48000))
    wav, sr = A.load_audio(path, 44100, dst_ch, device=DEV)
    want = A.convert_audio(torch.from_numpy(decode_oracle(payload, pcm, src_ch)).to(DEV), 48000, 44100, dst_ch)
    assert sr == 44100 and torch.equal(wav, want)


@pytest.mark.gpu
def test_gpu_separate_audio_file(tmp_path):
    """separate_audio_file on a 48 kHz mono s24 file against separate_tensor of the oracle's decode and against the
    oracle chain of test_gpu_separator_resamples_and_emits_pcm.  The decoded, converted wave is bitwise the same; the
    stems are compared within a bound because two forwards of one input differ in the last bits (GroupNorm partial
    sums meet through order-dependent atomics)."""
    import demucs_b200 as D
    from _fixtures import small_config, init_weights
    from oracle.apply_oracle import apply_model_oracle
    from oracle import audio_oracle as O
    cfg = small_config()
    model = D.HTDemucs.from_config(cfg, init_seed=0, layer_scale=0.5)
    sep = D.Separator(model, device=DEV, shifts=0)
    payload = s24_payload(0.3 * np.random.default_rng(8).standard_normal((1, 90000)))
    path = wav_file(tmp_path / "m.wav", payload, fmt_body(S24, 1, 48000))
    wav48 = torch.from_numpy(decode_oracle(payload, S24, 1))
    wav, stems = sep.separate_audio_file(path)
    dev_wav, dev_stems = sep.separate_tensor(wav48.to(DEV), sr=48000)
    assert wav.device.type == "cpu" and torch.equal(wav, dev_wav.cpu())
    x44 = O.convert_audio(wav48, 48000, 44100, 2)
    ref = x44.mean(0)
    x = (x44 - ref.mean()) / (ref.std() + 1e-8)
    with torch.no_grad():
        want = apply_model_oracle((init_weights(cfg, 0, layer_scale=0.5), cfg), x[None], shifts=0)[0]
    want = want * (ref.std() + 1e-8) + ref.mean()
    for i, s in enumerate(cfg.sources):
        got = stems[s]
        assert got.device.type == "cpu" and got.dtype == torch.float32 and got.shape == want[i].shape
        assert rel_l2(got, dev_stems[s].cpu()) < 1e-4 and rel_l2(got, want[i]) < 1e-4, s


@pytest.mark.gpu
def test_gpu_round_trip_through_save_audio(tmp_path):
    x = 0.45 * torch.randn(2, 20011, generator=torch.Generator().manual_seed(13))
    for bits, scale in ((16, 2 ** 15), (24, 2 ** 23)):
        path = tmp_path / f"r{bits}.wav"
        A.save_audio(x.to(DEV), path, 44100, clip="none", bits_per_sample=bits)
        ints = A.stems_to_pcm(x.to(DEV), "none", bits).t().double()
        wav, _ = A.load_audio(path, device=DEV)
        assert torch.equal(wav.cpu().double(), ints / scale)
    path = tmp_path / "f.wav"
    A.save_audio(x.to(DEV), path, 44100, clip="none", as_float=True)
    wav, sr = A.load_audio(path, device=DEV)
    assert sr == 44100 and torch.equal(wav.cpu(), x)
