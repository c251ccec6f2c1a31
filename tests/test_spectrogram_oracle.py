"""CPU checks of the float64 spectrogram-analysis restatement (tests/spectrogram_oracle.py) that the GPU kernel is
compared against, of the frame count the C ABI reports, and of ``audio.load_wav``."""
import ctypes as C
import os
import wave

import numpy as np
import pytest
import scipy.signal

import spectrogram_oracle as S
from oracle import audio_oracle as AO
from tacotron_multispeaker_b200.hparams import HParams

GOLD_AUDIO = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_audio.npz")


@pytest.mark.parametrize("L", [5000, 12345, 20001])
def test_stft_matches_scipy(L):
    """|librosa.stft| restated = |scipy.signal.stft| (boundary 'even' is np.pad's reflect; scipy divides by the window
    sum win/2) on the 1 + L // hop frames librosa keeps."""
    hp = HParams()
    n_fft, hop, win = AO.stft_parameters(hp)
    y = np.random.default_rng(L).standard_normal(L)
    got = np.abs(S.stft_librosa(y, n_fft, hop, win))
    _, _, Z = scipy.signal.stft(y, window="hann", nperseg=win, noverlap=win - hop, nfft=n_fft, boundary="even",
                                padded=False, detrend=False)
    T = 1 + L // hop
    assert got.shape == (T, n_fft // 2 + 1) and Z.shape[1] >= T
    want = np.abs(Z[:, :T].T) * (win / 2)
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(want)


def test_numpy_helpers_match_reference():
    """preemphasis, _amp_to_db and _normalize against the reference's own output."""
    g = np.load(GOLD_AUDIO)
    hp = HParams()
    np.testing.assert_allclose(S.preemphasis(g["x"], hp.preemphasis), g["preemphasis"], rtol=0, atol=1e-15)
    np.testing.assert_allclose(S.amp_to_db(g["amp"]), g["amp_to_db"], rtol=1e-14, atol=1e-12)
    np.testing.assert_allclose(S.normalize(AO.denormalize(g["spec"], hp) - 7.0, hp), g["normalize"], rtol=0, atol=1e-15)


def test_mel_scale_known_answers():
    assert float(S.hz_to_mel(1000.0)) == pytest.approx(15.0, abs=1e-12)
    assert float(S.hz_to_mel(500.0)) == pytest.approx(7.5, abs=1e-12)                       # linear part: 200/3 Hz per mel
    assert float(S.hz_to_mel(6400.0)) == pytest.approx(42.0, abs=1e-12)                      # log part: ln(6.4)/27 per mel
    f = np.array([0.0, 100.0, 999.0, 1000.0, 1001.0, 4321.0, 10000.0])
    np.testing.assert_allclose(S.mel_to_hz(S.hz_to_mel(f)), f, rtol=1e-13, atol=1e-10)


def test_mel_basis_known_answers():
    sr, n_fft, n_mels = 20000, 2048, 80
    M = S.mel_basis(sr, n_fft, n_mels)
    fft_f = np.linspace(0, sr / 2, n_fft // 2 + 1)
    mel_f = S.mel_frequencies(n_mels + 2, sr / 2)
    assert M.shape == (n_mels, 1025)
    assert mel_f[0] == 0.0 and mel_f[-1] == pytest.approx(sr / 2, rel=1e-12)
    df = sr / n_fft
    for i in range(n_mels):
        lo, c, hi = mel_f[i], mel_f[i + 1], mel_f[i + 2]
        inside = (fft_f > lo) & (fft_f < hi)
        assert np.all(M[i, ~inside] == 0.0), i                                   # zero outside (f_i, f_i+2)
        assert np.all(M[i, inside] > 0.0), i
        peak = 2.0 / (hi - lo)                                                    # triangle height after the scaling
        k = int(np.argmax(M[i]))
        assert abs(fft_f[k] - c) <= df, i                                         # the peak sits at the centre frequency
        assert M[i, k] <= peak * (1 + 1e-12)
        if hi - lo > 20 * df:                                                     # wide bands: unit area
            assert abs(M[i].sum() * df - 1.0) < 0.02, (i, M[i].sum() * df)
    U = S.mel_basis(sr, n_fft, n_mels, mel_scaled=False)
    assert U.max() == pytest.approx(1.0, abs=0.05) and np.allclose(M, U * (2.0 / (mel_f[2:] - mel_f[:-2]))[:, None])


@pytest.mark.parametrize("k0", [37, 100, 400])
def test_sinusoid_on_a_bin(k0):
    """A cosine of amplitude A on bin k0: |D| peaks at A win / 4 on interior frames (up to the leakage of the image
    at -k0), and the normalised spectrogram there is the formula of the reference applied to that amplitude, with
    the gain |1 - a exp(-i w)| of the pre-emphasis."""
    hp = HParams()
    n_fft, hop, win = AO.stft_parameters(hp)
    A, L = 0.7, 20000
    w = 2 * np.pi * k0 / n_fft
    y = A * np.cos(w * np.arange(L) + 0.3)
    D = np.abs(S.stft_librosa(y, n_fft, hop, win))
    interior = slice(5, 1 + L // hop - 5)
    assert np.all(np.argmax(D[interior], axis=1) == k0)
    np.testing.assert_allclose(D[interior, k0], A * win / 4, rtol=2e-3)
    gain = abs(1 - hp.preemphasis * np.exp(-1j * w))
    lin = S.spectrogram_librosa(y, hp)
    want = np.clip((20 * np.log10(A * gain * win / 4) - hp.ref_level_db - hp.min_level_db) / -hp.min_level_db, 0, 1)
    np.testing.assert_allclose(lin[interior, k0], want, atol=2e-4)


def test_reflect_padding_longer_than_the_signal():
    """np.pad(mode='reflect') with a pad longer than the signal is the even periodic extension of period 2 (L - 1);
    for L = 1 it repeats the sample (the index map the kernel uses)."""
    for L in (1, 2, 3, 7, 500):
        x = np.arange(1, L + 1, dtype=np.float64)
        got = np.pad(x, 1024, mode="reflect")
        j = np.arange(-1024, L + 1024)
        if L == 1:
            m = np.zeros_like(j)
        else:
            P = 2 * (L - 1)
            m = j % P
            m = np.where(m >= L, P - m, m)
        np.testing.assert_array_equal(got, x[m])


def test_spectrogram_frames_matches_librosa_frame_count():
    from tacotron_multispeaker_b200 import _abi
    from tacotron_multispeaker_b200.build import build_library
    build_library()
    lib = _abi.load()
    for fl, fs in ((50.0, 12.5), (50.0, 10.0), (49.95, 12.5), (102.4, 12.5)):
        hp = HParams(frame_length_ms=fl, frame_shift_ms=fs)
        ap = _abi.TacoAudioParams(hp.sample_rate, 0, fl, fs, hp.preemphasis, hp.min_level_db, hp.ref_level_db, hp.power)
        hop = AO.stft_parameters(hp)[1]
        for L in (1, 2, 249, 250, 251, 500, 1023, 5000, 20001, 250000, 10 ** 10):
            assert lib.taco_spectrogram_frames(C.byref(ap), L) == 1 + L // hop
        assert lib.taco_spectrogram_frames(C.byref(ap), 0) < 0
        ap.sample_rate = 0
        assert lib.taco_spectrogram_frames(C.byref(ap), 100) < 0


def _write_wav(path, pcm, rate, channels=1, width=2):
    with wave.open(str(path), "wb") as f:
        f.setnchannels(channels)
        f.setsampwidth(width)
        f.setframerate(rate)
        f.writeframes(pcm.tobytes())


def test_load_wav(tmp_path):
    from tacotron_multispeaker_b200 import audio
    pcm = np.array([0, 1, -1, 32767, -32768, 1234, -20000], "<i2")
    _write_wav(tmp_path / "a.wav", pcm, 20000)
    got = audio.load_wav(tmp_path / "a.wav", 20000)
    assert got.dtype == np.float32
    np.testing.assert_array_equal(got, pcm.astype(np.float32) / 32768)
    # save_wav's output reads back as its int16 samples / 32768
    wav = np.sin(np.arange(300) / 7.0) * 0.3
    audio.save_wav(wav, str(tmp_path / "b.wav"), 20000)
    np.testing.assert_array_equal(audio.load_wav(str(tmp_path / "b.wav"), 20000), audio.wav_to_int16(wav) / np.float32(32768))
    for name, rate, ch, width, data in (("sr.wav", 22050, 1, 2, pcm), ("st.wav", 20000, 2, 2, np.repeat(pcm, 2)),
                                        ("u8.wav", 20000, 1, 1, np.arange(7, dtype=np.uint8))):
        _write_wav(tmp_path / name, data, rate, ch, width)
        with pytest.raises(ValueError):
            audio.load_wav(tmp_path / name, 20000)


@pytest.mark.parametrize("mistake", ["symmetric padding", "pre-emphasis after padding", "window not centred",
                                     "mel bands not scaled"])
def test_each_convention_mistake_fails_the_accuracy_bound(mistake):
    """A kernel that made one of these mistakes would be off from the restatement by what the mistaken restatement
    is off by: on the seeded noise and chirp signals of the GPU accuracy test that exceeds the bound of that test by
    orders of magnitude."""
    hp = HParams()
    n_fft = AO.stft_parameters(hp)[0]
    M = S.mel_basis(hp.sample_rate, n_fft, hp.num_mels)
    kw = {"symmetric padding": dict(pad_mode="symmetric"), "pre-emphasis after padding": dict(preemph_after_pad=True),
          "window not centred": dict(lpad=0), "mel bands not scaled": dict(mel_scaled=False)}[mistake]
    for kind, L in (("noise", 5000), ("chirp", 20001), ("noise", 500)):
        y = S.make_signal(kind, L, 3).astype(np.float64)
        mags, s = S.magnitudes(y, hp), S.frame_abs_sum(y, hp)
        lin = S.normalize(S.amp_to_db(mags) - hp.ref_level_db, hp)
        mel = S.normalize(S.amp_to_db(mags @ M.T) - hp.ref_level_db, hp)
        if mistake == "mel bands not scaled":
            got, want, w, amp = S.melspectrogram_librosa(y, hp, **kw), mel, M.sum(axis=1), mags @ M.T
        else:
            got, want, w, amp = S.spectrogram_librosa(y, hp, **kw), lin, np.ones(mags.shape[1]), mags
        assert S.error_ratio(want, want, s, w, amp, hp) == 0.0
        assert S.error_ratio(got, want, s, w, amp, hp) > 100 * S.C_BOUND, (kind, L)
