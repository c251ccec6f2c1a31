"""float64 restatement of the reference's spectrogram analysis (util/audio.py spectrogram / melspectrogram) for the tests.

The numpy helpers (``preemphasis``, ``_amp_to_db``, ``_normalize``) are pinned to the reference's own output in
``tests/golden/ref_audio.npz``.  The two librosa 0.5.1 calls are restated here and stay unpinned against the library
(it is not installed):

* ``librosa.stft(y, n_fft, hop, win)`` with ``center=True``: ``y`` padded by ``n_fft / 2`` on both sides with
  ``np.pad(mode='reflect')``, ``1 + len(y) // hop`` frames of ``n_fft`` samples, the periodic Hann window of ``win``
  points centred in the frame (``lpad = (n_fft - win) // 2``), ``rfft``;
* ``librosa.filters.mel(sr, n_fft, n_mels)`` with fmin 0, fmax sr/2 and the Slaney mel scale; every triangle scaled by
  ``2 / (f[i+2] - f[i])`` (librosa 0.5 has no ``norm`` argument and always applies it).

The keyword switches (``pad_mode``, ``lpad``, ``preemph_after_pad``, ``mel_scaled``) restate deliberate mistakes; the
GPU tests use them to show that each mistake would be caught.
"""
from __future__ import annotations

import numpy as np

from oracle.audio_oracle import hann_periodic, stft_parameters


def preemphasis(x, a):
    """util/audio.py preemphasis: scipy.signal.lfilter([1, -a], [1], x)."""
    x = np.asarray(x, np.float64)
    y = x.copy()
    y[1:] -= a * x[:-1]
    return y


def amp_to_db(x):
    return 20.0 * np.log10(np.maximum(1e-5, x))


def normalize(S, hp):
    return np.clip((S - hp.min_level_db) / -hp.min_level_db, 0.0, 1.0)


def _rfft_frames(padded, T, n_fft, hop, win, lpad=None):
    window = np.zeros(n_fft)
    lp = (n_fft - win) // 2 if lpad is None else lpad
    window[lp:lp + win] = hann_periodic(win)
    idx = np.arange(n_fft)[None, :] + hop * np.arange(T)[:, None]
    return np.fft.rfft(padded[idx] * window[None, :], n_fft, axis=-1)


def stft_librosa(p, n_fft, hop, win, pad_mode="reflect", lpad=None):
    """librosa.stft(p, n_fft, hop, win) transposed to [1 + len(p) // hop, n_fft/2 + 1]."""
    p = np.asarray(p, np.float64)
    return _rfft_frames(np.pad(p, n_fft // 2, mode=pad_mode), 1 + len(p) // hop, n_fft, hop, win, lpad)


def frame_abs_sum(y, hp):
    """sum over each frame of |window * pre-emphasised sample|: the scale of that frame's fp32 transform error."""
    n_fft, hop, win = stft_parameters(hp)
    padded = np.pad(preemphasis(y, hp.preemphasis), n_fft // 2, mode="reflect")
    T = 1 + len(y) // hop
    lp = (n_fft - win) // 2
    idx = lp + np.arange(win)[None, :] + hop * np.arange(T)[:, None]
    return np.abs(padded[idx] * hann_periodic(win)[None, :]).sum(axis=1)


def hz_to_mel(f):
    f = np.asarray(f, np.float64)
    f_sp, min_log_hz, logstep = 200.0 / 3.0, 1000.0, np.log(6.4) / 27.0
    return np.where(f >= min_log_hz, min_log_hz / f_sp + np.log(np.maximum(f, 1e-300) / min_log_hz) / logstep, f / f_sp)


def mel_to_hz(m):
    m = np.asarray(m, np.float64)
    f_sp, min_log_hz, logstep = 200.0 / 3.0, 1000.0, np.log(6.4) / 27.0
    min_log_mel = min_log_hz / f_sp
    return np.where(m >= min_log_mel, min_log_hz * np.exp(logstep * (m - min_log_mel)), f_sp * m)


def mel_frequencies(n, fmax):
    return mel_to_hz(np.linspace(0.0, float(hz_to_mel(fmax)), n))


def mel_basis(sr, n_fft, n_mels, mel_scaled=True):
    """librosa.filters.mel(sr, n_fft, n_mels) (0.5.1): [n_mels, n_fft/2 + 1]."""
    fft_f = np.linspace(0.0, sr / 2.0, n_fft // 2 + 1)
    mel_f = mel_frequencies(n_mels + 2, sr / 2.0)
    fdiff = np.diff(mel_f)
    ramps = np.subtract.outer(mel_f, fft_f)
    w = np.zeros((n_mels, n_fft // 2 + 1))
    for i in range(n_mels):
        w[i] = np.maximum(0.0, np.minimum(-ramps[i] / fdiff[i], ramps[i + 2] / fdiff[i + 1]))
    if mel_scaled:
        w *= (2.0 / (mel_f[2:n_mels + 2] - mel_f[:n_mels]))[:, None]
    return w


def magnitudes(y, hp, pad_mode="reflect", lpad=None, preemph_after_pad=False):
    """|D| of util/audio.py _stft(preemphasis(y)), [frames, n_fft/2 + 1]."""
    n_fft, hop, win = stft_parameters(hp)
    y = np.asarray(y, np.float64)
    if preemph_after_pad:   # the mistake: filter the padded signal instead of padding the filtered one
        padded = preemphasis(np.pad(y, n_fft // 2, mode=pad_mode), hp.preemphasis)
        return np.abs(_rfft_frames(padded, 1 + len(y) // hop, n_fft, hop, win, lpad))
    return np.abs(stft_librosa(preemphasis(y, hp.preemphasis), n_fft, hop, win, pad_mode, lpad))


def spectrogram_librosa(y, hp, **mistakes):
    """util/audio.py spectrogram(y), transposed to [T, num_freq]."""
    return normalize(amp_to_db(magnitudes(y, hp, **mistakes)) - hp.ref_level_db, hp)


def melspectrogram_librosa(y, hp, mel_scaled=True, **mistakes):
    """util/audio.py melspectrogram(y), transposed to [T, num_mels]."""
    n_fft = stft_parameters(hp)[0]
    M = mel_basis(hp.sample_rate, n_fft, hp.num_mels, mel_scaled)
    return normalize(amp_to_db(magnitudes(y, hp, **mistakes) @ M.T) - hp.ref_level_db, hp)


# ---- the accuracy bound of the GPU tests ---------------------------------------------------------------------------
# An fp32 transform of a frame is off by at most c * sum|windowed frame| in every bin; through 20 log10 and the
# normalisation that is (20 / ln 10) / |min_level_db| * c * sum|frame| / max(1e-5, amplitude), plus 2^-22 for the
# log2 / fma rounding of the result.  The mel bands carry the sum of their weights as a factor.
# Measured on a B200 (1000 W limit) over every signal, length and geometry of tests/test_gpu_spectrogram.py: c = 2.05e-7
# at most (chirp, linear rows; the sine 1.35e-7, noise 2.4e-8, mel bands 1.7e-8, silence exact).  The bound is about 5x that.
C_BOUND = 1e-6


def error_ratio(got, want, frame_sum, weight_sum, amp, hp):
    """Largest (|got - want| - 2^-22) / ((20 / ln 10) / |min_level_db| * frame_sum * weight_sum / max(1e-5, amp)): the
    c an fp32 result needs to stay inside the bound.  inf where the bound is 0 (silent frames) and got != want."""
    got = np.asarray(got, np.float64)
    excess = np.maximum(np.abs(got - want) - 2.0 ** -22, 0.0)
    scale = (20.0 / np.log(10.0)) / abs(hp.min_level_db) * np.asarray(frame_sum)[:, None] * np.asarray(weight_sum)[None, :] \
        / np.maximum(1e-5, amp)
    ratio = np.where(scale > 0, excess / np.where(scale > 0, scale, 1.0), np.where(excess > 0, np.inf, 0.0))
    return float(ratio.max()) if ratio.size else 0.0


def reference_and_ratios(y, got_linear, got_mel, hp):
    """(c of the linear rows, c of the mel rows) of a kernel result for one utterance against this restatement."""
    n_fft = stft_parameters(hp)[0]
    M = mel_basis(hp.sample_rate, n_fft, hp.num_mels)
    mags = magnitudes(y, hp)
    s = frame_abs_sum(y, hp)
    lin = normalize(amp_to_db(mags) - hp.ref_level_db, hp)
    mel_amp = mags @ M.T
    mel = normalize(amp_to_db(mel_amp) - hp.ref_level_db, hp)
    return (error_ratio(got_linear, lin, s, np.ones(mags.shape[1]), mags, hp),
            error_ratio(got_mel, mel, s, M.sum(axis=1), mel_amp, hp))


def make_signal(kind, L, seed, sample_rate=20000):
    """Seeded float32 test signals: 'silence' (exact zeros), 'sine' (full scale, 440 Hz), 'noise', 'chirp'."""
    rng = np.random.default_rng(seed)
    t = np.arange(L) / sample_rate
    if kind == "silence":
        y = np.zeros(L)
    elif kind == "sine":
        y = 0.999 * np.sin(2 * np.pi * 440.0 * t + rng.uniform(0, 2 * np.pi))
    elif kind == "noise":
        y = rng.uniform(-0.5, 0.5, L)
    elif kind == "chirp":
        import scipy.signal
        y = 0.8 * scipy.signal.chirp(t, f0=60.0, t1=max(L / sample_rate, 1e-3), f1=9000.0) * (0.5 + 0.5 * rng.uniform())
    else:
        raise ValueError(kind)
    return y.astype(np.float32)
