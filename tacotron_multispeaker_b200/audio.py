"""Audio side of the synthesis surface: the parts of the reference's
``util/audio.py`` that ``Synthesizer.synthesize`` uses (``synthesizer.py:27,
47-56``), with the vocoder on the GPU.

* ``inv_spectrogram_tensorflow(engine, linear)`` -- reference
  ``util/audio.py:39-46,78-91`` (denormalise, dB -> amplitude, ``** power``,
  Griffin-Lim with ``tf.contrib.signal`` STFT conventions) as
  ``taco_griffin_lim`` kernels; batched over utterances.  Like the reference's
  it does NOT undo the pre-emphasis.
* ``synthesize_wav(engine, linear)`` -- the same followed by
  ``inv_preemphasis`` (``:23-24``), fused into the same call on the device.
* ``spectrogram(engine, wav)`` / ``melspectrogram(engine, wav)`` -- the
  analysis half (``preemphasis`` -> ``librosa.stft`` -> ``_amp_to_db`` ->
  ``_normalize``, and ``_linear_to_mel`` with ``librosa.filters.mel``) as the
  ``taco_spectrogram`` kernel.  They return ``[T, F]``, the layout the model
  and the feeder consume (the reference returns ``[F, T]`` and its
  preprocessing saves the transpose).
* ``resample(engine, y, orig_sr, target_sr)`` / ``load(engine, path,
  sample_rate)`` -- ``librosa.core.resample`` (resampy ``kaiser_best``,
  ``fix=True``) as the ``taco_resample`` kernel, and ``librosa.core.load``
  (16-bit PCM of any rate and channel count, mixed down on the host, resampled
  on the device): the reference reads its corpora with
  ``librosa.core.load(path, sr=hparams.sample_rate)``.
* ``save_wav`` (``:14-16``), ``load_wav``, ``find_endpoint`` (``:55-63``),
  ``_stft_parameters`` (``:114-118``) are host code (numpy / ``wave``): they
  handle a finished waveform once per utterance.

There is no CPU Griffin-Lim, STFT or resampler here: without the CUDA library these raise.
"""
from __future__ import annotations

import wave

import numpy as np


def _stft_parameters(hp):
    n_fft = (hp.num_freq - 1) * 2
    hop_length = int(hp.frame_shift_ms / 1000 * hp.sample_rate)
    win_length = int(hp.frame_length_ms / 1000 * hp.sample_rate)
    return n_fft, hop_length, win_length


def inv_spectrogram_tensorflow(engine, spectrogram, griffin_lim_iters=None):
    """Normalised linear spectrogram ``[T,num_freq]`` or ``[N,T,num_freq]`` (torch CUDA tensor or array) ->
    waveform(s) on the device, pre-emphasis not undone (the caller applies ``inv_preemphasis``)."""
    return engine.griffin_lim(spectrogram, griffin_lim_iters, inv_preemphasis=False)


def synthesize_wav(engine, spectrogram, griffin_lim_iters=None):
    """``inv_preemphasis(inv_spectrogram_tensorflow(x))`` in one device call (synthesizer.py:47-50)."""
    return engine.griffin_lim(spectrogram, griffin_lim_iters, inv_preemphasis=True)


def spectrogram(engine, wav):
    """Normalised linear spectrogram ``[T, num_freq]`` of one waveform (``[N, T, num_freq]`` for a batch or a list of
    waveforms), on the device."""
    return engine.spectrogram(wav)[0]


def melspectrogram(engine, wav):
    """Normalised mel spectrogram ``[T, num_mels]`` of one waveform (``[N, T, num_mels]`` for a batch or a list of
    waveforms), on the device."""
    return engine.spectrogram(wav)[1]


def load_wav(path, sample_rate):
    """Mono 16-bit PCM WAV file -> float32 samples in [-1, 1) (divided by 32768).  The reference's
    ``librosa.core.load(path, sr=sample_rate)`` also resamples and mixes down; that is not restated here, so any other
    sample rate, channel count or sample width raises ``ValueError``."""
    with wave.open(str(path), "rb") as f:
        if f.getframerate() != int(sample_rate) or f.getnchannels() != 1 or f.getsampwidth() != 2:
            raise ValueError("%s: need mono 16-bit PCM at %d Hz, got %d channel(s), %d-bit, %d Hz (no resampling here)"
                             % (path, int(sample_rate), f.getnchannels(), 8 * f.getsampwidth(), f.getframerate()))
        pcm = np.frombuffer(f.readframes(f.getnframes()), "<i2")
    return pcm.astype(np.float32) / np.float32(32768.0)


def resample(engine, y, orig_sr, target_sr):
    """``librosa.core.resample(y, orig_sr, target_sr)`` (``res_type='kaiser_best'``, ``fix=True``) of one waveform on the
    device: ``ceil(len(y) * target_sr / orig_sr)`` samples, the input unchanged when the rates are equal."""
    return engine.resample(y, orig_sr, target_sr)


def read_pcm(path):
    """librosa.core.load's samples before resampling, on the host: a 16-bit PCM WAV file as float32 ``pcm * (1 /
    32768)`` (audioread's conversion), channels mixed down with ``np.mean`` (``librosa.to_mono``).  Returns ``(samples,
    native rate)``.  Other sample widths raise ``ValueError``."""
    with wave.open(str(path), "rb") as f:
        channels, width, rate = f.getnchannels(), f.getsampwidth(), f.getframerate()
        if width != 2:
            raise ValueError("%s: need 16-bit PCM, got %d-bit" % (path, 8 * width))
        pcm = np.frombuffer(f.readframes(f.getnframes()), "<i2")
    y = np.float32(1.0 / 32768) * pcm.astype(np.float32)
    if channels > 1:
        y = np.mean(y.reshape((-1, channels)).T, axis=0)
    return y, rate


def load(engine, path, sample_rate):
    """``librosa.core.load(path, sr=sample_rate)`` for 16-bit PCM WAV files of any sample rate and channel count: read and
    mixed down on the host (``read_pcm``), resampled on the device (``resample``).  Returns a float32 CUDA tensor."""
    y, rate = read_pcm(path)
    if y.size == 0:
        raise ValueError("%s: no samples" % path)
    return engine.resample(y, rate, int(sample_rate))


def wav_to_int16(wav) -> np.ndarray:
    """The samples ``save_wav`` writes: peak-normalised to 32767 with the reference's 0.01 floor, truncated."""
    wav = np.asarray(wav, dtype=np.float32)
    wav = wav * np.float32(32767 / max(0.01, float(np.max(np.abs(wav))) if wav.size else 0.01))
    return wav.astype(np.int16)


def save_wav(wav, path, sample_rate):
    """Mono 16-bit PCM RIFF file, as ``librosa.output.write_wav`` produces for an int16 array."""
    pcm = wav_to_int16(wav)
    with wave.open(path, "wb") as f:
        f.setnchannels(1)
        f.setsampwidth(2)
        f.setframerate(int(sample_rate))
        f.writeframes(pcm.astype("<i2").tobytes())


def _db_to_amp(x):
    return np.power(10.0, x * 0.05)


def find_endpoint(wav, sample_rate, threshold_db=-10, min_silence_sec=2):
    wav = np.asarray(wav)
    window_length = int(sample_rate * min_silence_sec)
    hop_length = int(window_length / 4)
    threshold = _db_to_amp(threshold_db)
    for x in range(hop_length, len(wav) - window_length, hop_length):
        if np.max(wav[x:x + window_length]) < threshold:
            return x + hop_length
    return len(wav)
