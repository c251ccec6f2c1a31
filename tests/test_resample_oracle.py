"""CPU checks of the float64 restatement of librosa 0.5.1 resample / load with resampy's kaiser_best filter
(tests/resample_oracle.py) that the GPU kernel is compared against, of the length and the position replay the C ABI
reports, and of the host half of ``audio.load``."""
import wave

import numpy as np
import pytest
import scipy.special

import resample_oracle as R

RATES = [(8000, 20000), (11025, 20000), (16000, 20000), (22050, 20000), (24000, 20000), (44100, 20000),
         (48000, 20000), (20000, 16000), (44100, 16000)]


@pytest.fixture(scope="module")
def lib():
    from tacotron_multispeaker_b200 import _abi
    from tacotron_multispeaker_b200.build import build_library
    build_library()
    return _abi.load()


def test_filter_table():
    win = R.filter_table()
    assert win.size == 32769
    assert win[0] == R.ROLLOFF                                            # kaiser centre 1, sinc(0) = 1
    end = R.ROLLOFF * np.sinc(R.ROLLOFF * 64) / scipy.special.i0(R.BETA)   # the window's last point is 1 / I0(beta)
    assert win[-1] == pytest.approx(end, rel=1e-12, abs=1e-300)
    w_up, d_up = R.tables(16000, 20000)
    np.testing.assert_array_equal(w_up, win)                              # no scaling when upsampling
    w_dn, d_dn = R.tables(48000, 20000)
    np.testing.assert_array_equal(w_dn, win * (20000 / 48000))            # times the ratio when downsampling
    for w, d in ((w_up, d_up), (w_dn, d_dn)):
        assert d[-1] == 0.0
        np.testing.assert_array_equal(d[:-1], np.diff(w))
    assert R.index_step(48000, 20000) == 213 and R.index_step(22050, 20000) == 464 and R.index_step(16000, 20000) == 512


def _two_tone(sr):
    return lambda t: 0.5 * np.sin(2 * np.pi * 440.0 * t + 0.3) + 0.3 * np.sin(2 * np.pi * 0.3 * sr * t + 1.1)


@pytest.mark.parametrize("sr", [8000, 16000])
def test_upsampling_reproduces_in_band_tones(sr):
    f = _two_tone(sr)
    L = 2 * sr
    y = R.resample(f(np.arange(L) / sr), sr, 20000)
    assert y.size == 40000
    inner = slice(1000, y.size - 1000)                                    # away from the edges (64 zero crossings)
    err = np.abs(y[inner] - f(np.arange(y.size) / 20000)[inner]).max()
    assert err < 1e-6, err                                                # measured 5.1e-7 at both rates


@pytest.mark.parametrize("sr", [8000, 16000])
def test_upsampling_keeps_a_constant(sr):
    y = R.resample(np.ones(sr), sr, 20000)
    assert np.abs(y[1000:-1000] - 1.0).max() < 1e-7


@pytest.mark.parametrize("sr,dc", [(48000, 9.4817e-4), (22050, 1.2097e-4)])
def test_downsampling_dc_error_of_the_truncated_step(sr, dc):
    """index_step = int(scale * 512) (213 instead of 213.33 at 48 kHz) puts the DC gain of a downsampled constant off
    by this much: part of the reference's output."""
    y = R.resample(np.ones(2 * sr), sr, 20000)[2000:-2000]
    assert y.mean() - 1.0 == pytest.approx(dc, rel=2e-3)


def test_equal_rates_and_short_inputs():
    x = np.arange(5, dtype=np.float64)
    np.testing.assert_array_equal(R.resample(x, 20000, 20000), x)
    np.testing.assert_array_equal(R.resample(np.ones(1), 48000, 20000), [0.0])         # int(0.42) = 0 computed, ceil 1
    y = R.resample(np.ones(3), 16000, 20000)
    assert y.size == 4 and y[3] == 0.0 and np.all(y[:3] != 0.0)


def test_resample_length_matches_numpy(lib):
    cases = [(441, 22050, 400), (1, 48000, 20000), (3, 16000, 20000)]
    for L in (1, 2, 3, 4, 5, 7, 99, 100, 101, 441, 882, 12345, 60000, 250000, 600000, 10 ** 9):
        for so, sn in RATES + [(20000, 20000), (22050, 400), (48000, 1), (1, 7)]:
            cases.append((L, so, sn))
    for L, so, sn in cases:
        assert lib.taco_resample_length(L, so, sn) == int(np.ceil(L * (float(sn) / so))), (L, so, sn)
    assert lib.taco_resample_length(441, 22050, 400) == 8
    assert lib.taco_resample_length(1, 48000, 20000) == 1
    assert lib.taco_resample_length(3, 16000, 20000) == 4
    for L, so, sn in ((0, 16000, 20000), (-5, 16000, 20000), (10, 0, 20000), (10, 16000, -1)):
        assert lib.taco_resample_length(L, so, sn) < 0


@pytest.mark.parametrize("so,sn", RATES)
def test_positions_equal_the_register_replay(lib, so, sn):
    count = 250000
    n, ol, el, orr, er = (np.empty(count, np.int32), np.empty(count, np.int32), np.empty(count, np.float32),
                          np.empty(count, np.int32), np.empty(count, np.float32))
    assert lib.taco_resample_positions(so, sn, 0, count, *(a.ctypes.data for a in (n, ol, el, orr, er))) == 0
    pn, pol, pel, por, per = R.positions(so, sn, count)
    np.testing.assert_array_equal(n, pn)
    np.testing.assert_array_equal(ol, pol)
    np.testing.assert_array_equal(orr, por)
    np.testing.assert_array_equal(el, pel.astype(np.float32))
    np.testing.assert_array_equal(er, per.astype(np.float32))
    assert ol.min() >= 0 and ol.max() <= 512 and orr.min() >= 0 and orr.max() <= 512
    # a window further on is the same replay
    t0, k = 123457, 1000
    m = [np.empty(k, a.dtype) for a in (n, ol, el, orr, er)]
    assert lib.taco_resample_positions(so, sn, t0, k, *(a.ctypes.data for a in m)) == 0
    for got, want in zip(m, (n, ol, el, orr, er)):
        np.testing.assert_array_equal(got, want[t0:t0 + k])


def test_positions_refusals(lib):
    buf = [np.empty(4, d) for d in (np.int32, np.int32, np.float32, np.int32, np.float32)]
    ptrs = [a.ctypes.data for a in buf]
    assert lib.taco_resample_positions(0, 20000, 0, 4, *ptrs) < 0
    assert lib.taco_resample_positions(16000, -1, 0, 4, *ptrs) < 0
    assert lib.taco_resample_positions(16000, 20000, -1, 4, *ptrs) < 0
    assert lib.taco_resample_positions(16000, 20000, (1 << 24) - 2, 4, *ptrs) < 0     # the 2^24 cap
    assert lib.taco_resample_positions(16000, 20000, (1 << 24) - 4, 4, *ptrs) == 0


def test_accumulated_register_flips():
    """Where t q / p is an integer the accumulated register can land just below it: n drops by one and frac jumps to
    scale.  It happens at 48 and 22.05 kHz over the first 250 000 outputs."""
    for so in (48000, 22050):
        n = R.positions(so, 20000, 250000)[0]
        t = np.arange(250000, dtype=np.int64)
        assert np.any(n != t * so // 20000), so


@pytest.mark.parametrize("mistake", ["exact rational positions", "untruncated index_step", "int output length"])
def test_each_convention_mistake_fails_the_accuracy_bound(mistake):
    """A kernel that made one of these mistakes would be off from the restatement by what the mistaken restatement is
    off by: on seeded noise and chirps that exceeds the GPU bound by more than 100x.  A kernel writing int(L ratio)
    samples instead of ceil has the wrong output length, which the GPU tests check."""
    for so, kind, L in ((48000, "noise", 60001), (22050, "chirp", 44101), (48000, "chirp", 30001), (22050, "noise", 22051)):
        x = R.make_signal(kind, L, 7, so).astype(np.float64)
        want, s = R.resample_f(x, so, 20000, with_abs=True)
        assert R.error_ratio(want, want, s) == 0.0
        if mistake == "int output length":
            assert len(R.resample(x, so, 20000, length="int")) != len(R.resample(x, so, 20000)), (so, L)
            continue
        kw = {"exact rational positions": dict(exact_positions=True), "untruncated index_step": dict(exact_step=True)}[mistake]
        got = R.resample_f(x, so, 20000, **kw)
        assert R.error_ratio(got, want, s) > 100 * R.C_BOUND, (so, kind, L)


def _write_wav(path, frames, rate, channels, width):
    with wave.open(str(path), "wb") as f:
        f.setnchannels(channels)
        f.setsampwidth(width)
        f.setframerate(rate)
        f.writeframes(frames)


@pytest.mark.parametrize("channels", [1, 2, 3])
def test_load_host_half_mixes_down_with_np_mean(tmp_path, channels):
    from tacotron_multispeaker_b200 import audio
    rng = np.random.default_rng(channels)
    pcm = rng.integers(-32768, 32768, size=(1001, channels)).astype("<i2")
    pcm[:3] = [[32767] * channels, [-32768] * channels, [0] * channels]
    _write_wav(tmp_path / "a.wav", pcm.tobytes(), 44100, channels, 2)
    y, rate = audio.read_pcm(tmp_path / "a.wav")
    assert rate == 44100 and y.dtype == np.float32 and y.shape == (1001,)
    f = pcm.astype(np.float32) * np.float32(1.0 / 32768)
    want = f[:, 0] if channels == 1 else np.mean(f.T, axis=0)
    np.testing.assert_array_equal(y, want)
    np.testing.assert_array_equal(y, R.pcm_to_float(pcm.reshape(-1), channels))
    if channels == 1:
        np.testing.assert_array_equal(y, pcm[:, 0].astype(np.float32) / 32768)    # load_wav's conversion, bit for bit


@pytest.mark.parametrize("width", [1, 3])
def test_load_refuses_other_sample_widths(tmp_path, width):
    from tacotron_multispeaker_b200 import audio
    _write_wav(tmp_path / "b.wav", bytes(range(6 * width)), 16000, 1, width)
    with pytest.raises(ValueError):
        audio.read_pcm(tmp_path / "b.wav")
