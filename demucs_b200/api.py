"""``Separator`` -- user-facing front door (drop-in for reference demucs/api.py:53-319).

Keeps the reference's constructor, ``update_parameter``, ``separate_tensor`` and the
``samplerate / audio_channels / model`` properties.  A model name / signature is resolved as in the
reference (``demucs_b200.repo.get_model``: a local ``repo`` folder of ``.th`` packages and bag YAML files,
or the remote zoo as far as torch hub has it cached -- there is no network here); ``"synthetic:<name>"``
names the random-init stand-ins of the released architectures, and a model object can be passed directly.
Audio that is not at the model's sample rate / channel count is converted on the device
(``demucs_b200.audio.convert_audio``, the julius-equivalent polyphase resampler), and
``separate_tensor_pcm`` / ``demucs_b200.audio.save_audio`` take the stems off the GPU in wire format
(clip prevention + PCM quantisation as device kernels).  ``separate_audio_file`` decodes RIFF/WAVE files on the
device (``demucs_b200.audio.load_audio``) and separates them there; other files still go through ``torchaudio``.
"""
from __future__ import annotations

from pathlib import Path
from typing import Callable, Dict, Optional, Tuple, Union

import torch as th

from .apply import apply_model, BagOfModels, _replace_dict
from .hdemucs import HDemucs
from .htdemucs import HTDemucs, htdemucs


class LoadAudioError(Exception):
    pass


class LoadModelError(Exception):
    pass


class _NotProvided:
    pass


NotProvided = _NotProvided()

SOURCES_4 = ["drums", "bass", "other", "vocals"]


def _builtin(name: str):
    """Random-init stand-ins for the released checkpoints (remote/*.yaml): ``synthetic:<name>``."""
    if name == "htdemucs":
        return htdemucs(SOURCES_4)
    if name == "htdemucs_6s":
        return htdemucs(SOURCES_4 + ["guitar", "piano"])
    if name == "htdemucs_ft":  # bag of 4 fine-tuned models, one per source (remote/htdemucs_ft.yaml)
        models = [htdemucs(SOURCES_4, init_seed=i) for i in range(4)]
        weights = [[1. if k == i else 0. for k in range(4)] for i in range(4)]
        return BagOfModels(models, weights)
    return None


def list_models(repo: Optional[Path] = None) -> Dict[str, Dict[str, Union[str, Path]]]:
    """Reference api.py:322-346: the single models and the bags of a repo (default: the HTDemucs part of the remote zoo)."""
    from .repo import RemoteRepo, LocalRepo, BagOnlyRepo
    model_repo = RemoteRepo() if repo is None else LocalRepo(Path(repo))
    bag_repo = BagOnlyRepo(None if repo is None else Path(repo), model_repo)
    return {"single": dict(model_repo.list_model()), "bag": dict(bag_repo.list_model())}


class Separator:
    def __init__(
        self,
        model: Union[str, HTDemucs, HDemucs, BagOfModels] = "htdemucs",
        repo: Optional[Path] = None,
        device: str = "cuda" if th.cuda.is_available() else "cpu",
        shifts: int = 1,
        overlap: float = 0.25,
        split: bool = True,
        segment: Optional[int] = None,
        jobs: int = 0,
        progress: bool = False,
        callback: Optional[Callable[[dict], None]] = None,
        callback_arg: Optional[dict] = None,
    ):
        """Same parameters as the reference ``Separator`` (api.py:54-116); ``model`` may also be a
        model object.  See ``apply_model`` for ``shifts / overlap / split / segment / callback``."""
        self._name = model
        self._repo = repo
        self._load_model()
        self.update_parameter(device=device, shifts=shifts, overlap=overlap, split=split,
                              segment=segment, jobs=jobs, progress=progress, callback=callback,
                              callback_arg=callback_arg)

    def update_parameter(self, device=NotProvided, shifts=NotProvided, overlap=NotProvided, split=NotProvided,
                         segment=NotProvided, jobs=NotProvided, progress=NotProvided, callback=NotProvided,
                         callback_arg=NotProvided):
        """Reference api.py:118-197."""
        for name, value in (("device", device), ("shifts", shifts), ("overlap", overlap), ("split", split),
                            ("segment", segment), ("jobs", jobs), ("progress", progress),
                            ("callback", callback), ("callback_arg", callback_arg)):
            if not isinstance(value, _NotProvided):
                setattr(self, "_" + name, value)

    def _load_model(self):
        if isinstance(self._name, (HTDemucs, HDemucs, BagOfModels)):
            self._model = self._name
        elif isinstance(self._name, str) and self._name.startswith("synthetic:"):
            self._model = _builtin(self._name[len("synthetic:"):])
        else:
            from .repo import get_model, ModelLoadingError
            try:
                self._model = get_model(name=self._name, repo=self._repo)      # api.py:199-201
            except ModelLoadingError as err:
                raise LoadModelError(f"Failed to load model: {err}") from err
        if self._model is None:
            raise LoadModelError("Failed to load model")
        self._audio_channels = self._model.audio_channels
        self._samplerate = self._model.samplerate

    def _load_audio(self, track: Path):
        """The reference's ``_load_audio`` with the device WAV decoder in place of ffmpeg: a RIFF/WAVE file comes back on
        ``self._device`` at the model's rate and channel count; anything it cannot decode goes to torchaudio."""
        from .audio import load_audio
        errors = {}
        try:
            return load_audio(track, self._samplerate, self._audio_channels, device=self._device)[0]
        except Exception as err:  # noqa
            errors["demucs_b200.audio.load_audio"] = err
        try:
            import torchaudio as ta
            wav, sr = ta.load(str(track))
        except Exception as err:  # noqa
            errors["torchaudio"] = err
            raise LoadAudioError("\n".join(f"When trying to load using {backend}, got the following error: {error}"
                                           for backend, error in errors.items()))
        if sr != self._samplerate or wav.shape[0] != self._audio_channels:      # api.py:221: convert_audio, on the device
            from .audio import convert_audio
            wav = convert_audio(wav.to(self._device), sr, self._samplerate, self._audio_channels).cpu()
        return wav

    def separate_tensor(self, wav: th.Tensor, sr: Optional[int] = None) -> Tuple[th.Tensor, Dict[str, th.Tensor]]:
        """Reference api.py:241-291: normalise by the mono mean/std, separate, de-normalise.
        ``wav`` [channels, length] float32 is modified in place and restored, as in the reference."""
        home = wav.device
        if sr is not None and sr != self.samplerate:        # api.py:265-266, as a device kernel
            from .audio import convert_audio
            wav = convert_audio(wav.to(self._device), sr, self._samplerate, self._audio_channels).to(home)
        ref = wav.mean(0)
        wav -= ref.mean()
        wav /= ref.std() + 1e-8
        out = apply_model(
            self._model,
            wav[None],
            segment=self._segment,
            shifts=self._shifts,
            split=self._split,
            overlap=self._overlap,
            device=self._device,
            num_workers=self._jobs,
            callback=self._callback,
            callback_arg=_replace_dict(self._callback_arg, ("audio_length", wav.shape[1])),
            progress=self._progress,
        )
        if out is None:
            raise KeyboardInterrupt
        out *= ref.std() + 1e-8
        out += ref.mean()
        wav *= ref.std() + 1e-8
        wav += ref.mean()
        return (wav, dict(zip(self._model.sources, out[0])))

    def separate_tensor_pcm(self, wav: th.Tensor, sr: Optional[int] = None, clip: Optional[str] = "rescale",
                            bits_per_sample: int = 16, as_float: bool = False) -> Dict[str, th.Tensor]:
        """``separate_tensor`` with the back door of ``save_audio`` (audio.py:236-265) attached, device-resident end to
        end: the wave is converted / normalised / separated on the GPU and every stem leaves it as interleaved PCM
        frames [frames, channels] (int16, 24-bit in int32, or float32) in pinned host memory -- clip prevention and
        quantisation are device kernels, so a 16-bit stem costs half the PCIe bytes of a float one."""
        from .audio import stems_to_pcm
        dev_wav = wav.to(self._device, copy=True)
        _, stems = self.separate_tensor(dev_wav, sr)
        return {name: stems_to_pcm(stem, clip, bits_per_sample, as_float) for name, stem in stems.items()}

    def separate_audio_file(self, file: Path):
        """As the reference: ``(wav, {stem: tensor})`` on the host.  A WAV file is decoded, converted and
        separated on the device; the wave and the stems come to the host at the end."""
        wav, stems = self.separate_tensor(self._load_audio(file), self.samplerate)
        return wav.cpu(), {name: stem.cpu() for name, stem in stems.items()}

    @property
    def samplerate(self):
        return self._samplerate

    @property
    def audio_channels(self):
        return self._audio_channels

    @property
    def model(self):
        return self._model
