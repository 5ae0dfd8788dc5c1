"""ORACLE -- TEST INFRASTRUCTURE ONLY.

Generates tests/golden/*.npz by running the UNMODIFIED reference (imported read-only
from /root/reference through oracle/refload.py) on the synthetic fixtures.  Run in the
build container:  ``python -m oracle.make_golden``.  The GPU box has no reference tree;
the committed .npz files are what pins the oracle and the CUDA path there.

Large tensors are stored as strided samples (the stride is stored next to them).
"""
from __future__ import annotations

import os
import random
from fractions import Fraction

import numpy as np
import torch

from demucs_b200.config import HTDemucsConfig, htdemucs_config
from demucs_b200.weights import init_weights
from . import refload

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def small_config() -> HTDemucsConfig:
    """Same topology as htdemucs, thin enough for the CPU oracle to finish in < 1 s."""
    cfg = HTDemucsConfig(sources=["a", "b", "c"], channels=16, dconv_mode=3, bottom_channels=128,
                         t_heads=2, t_layers=5, segment=Fraction(3, 2))
    cfg.validate()
    return cfg


def synth_mix(batch: int, length: int, seed: int, channels: int = 2) -> torch.Tensor:
    """White noise + a few partials so that the spectrum is not flat (SURVEY.md 8d)."""
    g = torch.Generator().manual_seed(seed)
    x = 0.1 * torch.randn(batch, channels, length, generator=g)
    t = torch.arange(length, dtype=torch.float64) / 44100.0
    for k, f in enumerate((110.0, 440.0, 1760.0)):
        x += (0.05 / (k + 1)) * torch.sin(2 * np.pi * f * t + k).float()
    x += 0.01  # DC offset so that the mean subtraction paths are exercised
    return x


def sample(x: torch.Tensor, stride: int) -> np.ndarray:
    return x.detach().reshape(-1)[::stride].float().numpy().copy()


def reference_taps(model, mix):
    """Forward with hooks on the reference's own sub-modules -> (out, taps in NCHW)."""
    taps = {}
    hooks = []

    def grab(name, fn=lambda o: o):
        def hook(_m, _i, o):
            taps[name] = fn(o).detach()
        return hook

    for i in range(4):
        hooks.append(model.encoder[i].register_forward_hook(grab(f"enc{i}")))
        hooks.append(model.tencoder[i].register_forward_hook(grab(f"tenc{i}")))
        hooks.append(model.decoder[i].register_forward_hook(grab(f"dec{i}", lambda o: o[0])))
        hooks.append(model.tdecoder[i].register_forward_hook(grab(f"tdec{i}", lambda o: o[0])))
    ct = model.crosstransformer
    for i in range(len(ct.layers)):
        hooks.append(ct.layers[i].register_forward_hook(grab(f"xf.layer{i}")))
        hooks.append(ct.layers_t[i].register_forward_hook(grab(f"xt.layer{i}")))
    with torch.no_grad():
        out = model(mix)
        z = model._spec(torch.nn.functional.pad(
            mix, (0, int(model.segment * model.samplerate) - mix.shape[-1])))
        taps["stft"] = model._magnitude(z)
        frs = torch.arange(taps["enc0"].shape[-2])
        emb = model.freq_emb(frs).t()[None, :, :, None]
        taps["enc0"] = taps["enc0"] + model.freq_emb_scale * emb
    for h in hooks:
        h.remove()
    B, D, Fr, T1 = out.shape[0], ct.layers[0].linear2.out_features, 8, taps["stft"].shape[-1]
    for i in range(len(ct.layers)):
        taps[f"xf.layer{i}"] = taps[f"xf.layer{i}"].view(B, T1, Fr, D).permute(0, 3, 2, 1)
        taps[f"xt.layer{i}"] = taps[f"xt.layer{i}"].transpose(1, 2)
    return out, taps


def forward_fixture(name, cfg, seed, layer_scale, batch, length, stride, tap_stride):
    W = init_weights(cfg, seed, layer_scale=layer_scale)
    model = refload.build_reference_model(cfg, W)
    mix = synth_mix(batch, length, 1234 + seed)
    out, taps = reference_taps(model, mix)
    data = {"out": sample(out, stride), "stride": stride, "tap_stride": tap_stride,
            "seed": seed, "layer_scale": -1.0 if layer_scale is None else layer_scale,
            "batch": batch, "length": length, "out_shape": np.array(out.shape),
            "out_norm": float(out.double().norm())}
    for k, v in taps.items():
        data[f"tap.{k}"] = sample(v, tap_stride)
        data[f"tapnorm.{k}"] = float(v.double().norm())
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), **data)
    print(name, {k: (v.shape if hasattr(v, "shape") else v) for k, v in data.items() if k in ("out",)})


APPLY_CASES = {
    "split": dict(shifts=0, split=True, overlap=0.25),
    "shifts2": dict(shifts=2, split=True, overlap=0.25),
    "power2": dict(shifts=1, split=True, overlap=0.1, transition_power=2.0),
    "segment1": dict(shifts=0, split=True, overlap=0.25, segment=1.0),
    "nosplit": dict(shifts=0, split=False),
}
BAG_WEIGHTS = [[1.0, 0.0, 0.5], [0.0, 1.0, 0.5]]


def apply_fixture(stride=23):
    ref = refload.load()
    cfg = small_config()
    Ws = [init_weights(cfg, s, layer_scale=0.5) for s in range(2)]
    models = [refload.build_reference_model(cfg, W) for W in Ws]
    mix = synth_mix(1, int(44100 * 3.3), 99)
    data = {"stride": stride, "length": mix.shape[-1]}
    for name, kw in APPLY_CASES.items():
        m = mix[..., :50000] if name == "nosplit" else mix
        random.seed(0)
        data[name] = sample(ref.apply_model(models[0], m.clone(), **kw), stride)
    random.seed(0)
    bag = ref.BagOfModels(models, weights=BAG_WEIGHTS)
    data["bag"] = sample(ref.apply_model(bag, mix.clone(), shifts=1), stride)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "apply_small.npz"), **data)
    print("apply_small", list(data))


def spectral_fixture():
    """``_spec``/``_magnitude`` and ``_mask``/``_ispec`` of the reference on their own."""
    ref = refload.load()
    model = ref.HTDemucs(sources=["a", "b"], segment=Fraction(39, 5)).eval()
    data = {}
    for name, L in (("full", 343980), ("odd", 50001)):
        x = synth_mix(2, L, 7)
        with torch.no_grad():
            mag = model._magnitude(model._spec(x))
            g = torch.Generator().manual_seed(11)
            spec = torch.randn(2, 2, 4, 2048, mag.shape[-1], generator=g)
            wav = model._ispec(model._mask(None, spec), L)
        data[f"{name}.stft"] = sample(mag, 97)
        data[f"{name}.stft_shape"] = np.array(mag.shape)
        data[f"{name}.istft"] = sample(wav, 31)
        data[f"{name}.istft_shape"] = np.array(wav.shape)
    np.savez_compressed(os.path.join(GOLDEN_DIR, "spectral.npz"), **data)
    print("spectral", {k: v.shape for k, v in data.items()})


def core_fixture():
    """``HTDemucs.forward_core`` of the reference (htdemucs.py:662-759) on the small geometry; the spectrogram handed in
    is the mixture's own plus noise, so that the result depends on the ``mag`` argument and not on a recomputed STFT."""
    cfg = small_config()
    W = init_weights(cfg, 0, layer_scale=0.5)
    model = refload.build_reference_model(cfg, W)
    mix = synth_mix(2, cfg.segment_length, 1240)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        mag = model._magnitude(model._spec(mix))
        mag = mag + 0.05 * mag.std() * torch.randn(mag.shape, generator=g)
        spec_out, time_out = model.forward_core(mag, mix)
    data = {"spec_out": sample(spec_out, 211), "time_out": sample(time_out, 7), "spec_shape": np.array(spec_out.shape),
            "time_shape": np.array(time_out.shape), "mag": sample(mag, 211)}
    np.savez_compressed(os.path.join(GOLDEN_DIR, "core_small.npz"), **data)
    print("core_small", {k: v.shape for k, v in data.items()})


def inventory_fixture():
    """Key order and shapes of the reference's ``HTDemucs.state_dict()`` on the small geometry."""
    ref = refload.load()
    sd = ref.HTDemucs(**small_config().reference_kwargs()).state_dict()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "small_inventory.npz"), names=np.array(list(sd)),
                        shapes=np.array([str(tuple(v.shape)) for v in sd.values()]))
    print("small_inventory", len(sd), "tensors")


def hdemucs_reference(cfg, W):
    refload.load()
    import demucs.hdemucs as H
    model = H.HDemucs(**cfg.reference_kwargs()).eval()
    model.load_state_dict({k: v.float() for k, v in W.items()}, strict=True)
    return model


def hdemucs_fixture(name, cfg, seed, layer_scale, batch, length, stride, tap_stride):
    """``HDemucs.forward`` of the reference (hdemucs.py:689-794) with hooks on every encoder / decoder layer."""
    from demucs_b200.hdemucs import init_weights as h_init
    W = h_init(cfg, seed, layer_scale)
    model = hdemucs_reference(cfg, W)
    mix = synth_mix(batch, length, 4321 + seed)
    taps, hooks = {}, []

    def grab(key, fn=lambda o: o):
        def hook(_m, _i, o):
            taps[key] = fn(o).detach()
        return hook
    for i in range(len(model.encoder)):
        hooks.append(model.encoder[i].register_forward_hook(grab(f"enc{i}")))
        hooks.append(model.decoder[i].register_forward_hook(grab(f"dec{i}", lambda o: o[0])))
    for i in range(len(model.tencoder)):
        hooks.append(model.tencoder[i].register_forward_hook(grab(f"tenc{i}")))
        hooks.append(model.tdecoder[i].register_forward_hook(grab(f"tdec{i}", lambda o: o[0])))
    with torch.no_grad():
        out = model(mix)
        frs = torch.arange(taps["enc0"].shape[-2])
        taps["enc0"] = taps["enc0"] + model.freq_emb_scale * model.freq_emb(frs).t()[None, :, :, None]
    for h in hooks:
        h.remove()
    data = {"out": sample(out, stride), "stride": stride, "tap_stride": tap_stride, "seed": seed,
            "layer_scale": -1.0 if layer_scale is None else layer_scale, "batch": batch, "length": length,
            "out_shape": np.array(out.shape), "names": np.array(list(W)), "shapes": np.array([str(tuple(v.shape)) for v in W.values()])}
    for k, v in taps.items():
        data[f"tap.{k}"] = sample(v, tap_stride)
    np.savez_compressed(os.path.join(GOLDEN_DIR, name), **data)
    print(name, data["out"].shape, len(taps), "taps")


def hdemucs_small_config():
    """The hdemucs_mmi topology (6 layers, GroupNorm / BLSTM / LocalState from layer 4, inject at layer 4), thin."""
    from demucs_b200.hdemucs import HDemucsConfig
    cfg = HDemucsConfig(sources=["a", "b", "c"], channels=16, dconv_comp=4, dconv_init=1e-3, segment=3)
    cfg.validate()
    return cfg


def audio_fixture():
    """The reference's own ``convert_audio_channels`` / ``prevent_clip`` / ``i16_pcm`` (audio.py:143-166,175-180,218-233;
    lameenc is stubbed: it only serves mp3 encoding) on fixed inputs."""
    import sys
    import types
    refload.load()
    sys.modules.setdefault("lameenc", types.ModuleType("lameenc"))
    import demucs.audio as ra
    g = torch.Generator().manual_seed(21)
    data = {}
    x5 = torch.randn(3, 5, 1000, generator=g)
    data["ch_5to2"] = ra.convert_audio_channels(x5, 2).contiguous().numpy()
    data["ch_5to1"] = ra.convert_audio_channels(x5, 1).contiguous().numpy()
    data["ch_1to2"] = ra.convert_audio_channels(x5[:, :1], 2).contiguous().numpy()
    loud = 1.7 * torch.randn(2, 5000, generator=g)
    quiet = 0.2 * torch.randn(2, 5000, generator=g)
    for mode in ("rescale", "clamp", "tanh"):
        data[f"clip_{mode}_loud"] = ra.prevent_clip(loud.clone(), mode).numpy()
        data[f"clip_{mode}_quiet"] = ra.prevent_clip(quiet.clone(), mode).numpy()
    data["i16_loud"] = ra.i16_pcm(loud.clone()).numpy()
    np.savez_compressed(os.path.join(GOLDEN_DIR, "audio.npz"), **data)
    print("audio", {k: v.shape for k, v in data.items()})


def main():
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    torch.set_num_threads(8)
    spectral_fixture()
    small = small_config()
    forward_fixture("small_ls05.npz", small, 0, 0.5, 2, small.segment_length, 7, 211)
    forward_fixture("small_short.npz", small, 1, 0.5, 1, 40001, 7, 211)
    full = htdemucs_config()
    forward_fixture("htdemucs_default.npz", full, 0, None, 1, full.segment_length, 29, 4999)
    forward_fixture("htdemucs_ls05.npz", full, 0, 0.5, 1, full.segment_length, 29, 4999)
    apply_fixture()
    inventory_fixture()
    core_fixture()
    audio_fixture()
    from demucs_b200.hdemucs import hdemucs_mmi_config
    hdemucs_fixture("hdemucs_small.npz", hdemucs_small_config(), 0, 0.5, 2, 343980, 13, 211)
    hdemucs_fixture("hdemucs_small_odd.npz", hdemucs_small_config(), 1, 0.5, 1, 100001, 13, 211)
    hdemucs_fixture("hdemucs_mmi.npz", hdemucs_mmi_config(), 0, 0.5, 1, 343980, 29, 4999)


if __name__ == "__main__":
    main()
