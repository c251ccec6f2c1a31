"""Resampling on the GPU (taco_resample, Engine.resample, audio.resample / audio.load, the torch op,
Synthesizer.teacher_forced from recordings at other rates) against the float64 restatement of librosa 0.5.1
core.resample with resampy's kaiser_best filter (tests/resample_oracle.py).

Accuracy: per output, |got - want| <= c * sum |w| |x| + 2^-24 |want| with c = resample_oracle.C_BOUND; outputs the
filter does not compute (fix_length's tail, rows past their length) are exact zeros."""
import ctypes as C
import math
import wave

import numpy as np
import pytest
import torch

import resample_oracle as R
import spectrogram_oracle as S

pytestmark = pytest.mark.gpu

RATES = [(8000, 20000), (11025, 20000), (16000, 20000), (22050, 20000), (24000, 20000), (44100, 20000),
         (48000, 20000), (20000, 16000), (44100, 16000)]
MEASURED = {}   # worst c per case, printed at the end of the module


@pytest.fixture(scope="module")
def eng():
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    e = Engine(HParams(), id_num=0)       # resampling needs no weights
    yield e
    e.close()
    if MEASURED:
        print("\nresample c measured: " + ", ".join("%s %.3g" % kv for kv in sorted(MEASURED.items())))


def lengths_for(so, sn, long_signal):
    q = so // math.gcd(so, sn)            # input samples per period of the phase pattern
    L = [1, 2, 3, max(1, q - 1), q, q + 1, 300, 5 * so]
    return L + [int(12.5 * so)] if long_signal else L


def check_batch(e, xs, so, sn, tag):
    y, out_len = e.resample(xs, so, sn)
    torch.cuda.synchronize()
    want_len = [R.output_length(len(x), so, sn) for x in xs]
    assert list(out_len) == want_len and y.shape == (len(xs), max(want_len))
    y = y.cpu().numpy()
    worst = 0.0
    for i, x in enumerate(xs):
        computed = int(len(x) * (float(sn) / so))
        want, s = R.resample_f(x.astype(np.float64), so, sn, with_abs=True)
        c = R.error_ratio(y[i, :computed], want, s)
        worst = max(worst, c)
        assert c <= R.C_BOUND, (tag, len(x), c)
        assert not y[i, computed:].any(), (tag, len(x))        # fix_length's zero and the rows' padding
    MEASURED[tag] = worst


@pytest.mark.parametrize("so,sn", RATES)
@pytest.mark.parametrize("kind", ["silence", "sine", "noise", "chirp"])
def test_accuracy_against_float64(eng, so, sn, kind):
    xs = [R.make_signal(kind, L, 10 + i, so) for i, L in enumerate(lengths_for(so, sn, kind in ("noise", "chirp")))]
    check_batch(eng, xs, so, sn, "%s %d->%d" % (kind, so, sn))
    if kind == "silence":
        assert not eng.resample(xs, so, sn)[0].any()


def test_batch_equals_single_calls_and_repeats(eng):
    so, sn = 22050, 20000
    xs = [R.make_signal("chirp", L, 70 + i, so) for i, L in enumerate([7777, 441, 1, 50001, 3])]
    y, out_len = eng.resample(xs, so, sn)
    y2, _ = eng.resample(xs, so, sn)
    assert torch.equal(y, y2)
    for i, x in enumerate(xs):
        one = eng.resample(x, so, sn)
        assert one.shape == (out_len[i],) == (eng.resample_length(len(x), so, sn),)
        assert torch.equal(y[i, :out_len[i]], one)
    dense = np.zeros((5, 50001), np.float32)
    for i, x in enumerate(xs):
        dense[i, :len(x)] = x
    yd, ld = eng.resample(dense, so, sn, lengths=[len(x) for x in xs])
    assert torch.equal(yd, y) and list(ld) == list(out_len)
    # a rate pair in between rebuilds the tables; coming back gives the same bits
    eng.resample(xs[0], 48000, 20000)
    assert torch.equal(eng.resample(xs, so, sn)[0], y)


def test_equal_rates_copy(eng):
    xs = [R.make_signal("noise", L, 3 + i, 20000) for i, L in enumerate([1000, 1, 777])]
    y, out_len = eng.resample(xs, 20000, 20000)
    assert list(out_len) == [1000, 1, 777]
    y = y.cpu().numpy()
    for i, x in enumerate(xs):
        np.testing.assert_array_equal(y[i, :len(x)], x)
        assert not y[i, len(x):].any()


def test_nothing_written_outside_the_output(eng):
    so, sn = 48000, 20000
    xs = [R.make_signal("noise", L, 90 + i, so) for i, L in enumerate([12000, 1, 2345, 12])]
    dense = np.zeros((4, 12000), np.float32)
    for i, x in enumerate(xs):
        dense[i, :len(x)] = x
    lengths = np.array([len(x) for x in xs], np.int32)
    G = 4096
    x_dev = torch.from_numpy(dense).to(eng.device)
    for s, n in ((so, sn), (sn, sn)):
        want, _ = eng.resample(dense, s, n, lengths=lengths)
        L_out = want.shape[1] + 3                                # longer than the longest row's output
        buf = torch.full((2 * G + 4 * L_out,), float("nan"), device=eng.device)
        eng._ck(eng.lib.taco_resample(eng._h, s, n, C.c_void_p(x_dev.data_ptr()), lengths.ctypes.data, 4, 12000,
                                      C.c_void_p(buf.data_ptr() + 4 * G), L_out, eng.stream))
        torch.cuda.synchronize()
        assert torch.isnan(buf[:G]).all() and torch.isnan(buf[-G:]).all()
        got = buf[G:-G].view(4, L_out)
        assert torch.equal(got[:, :want.shape[1]], want) and not got[:, want.shape[1]:].any()


def test_torch_op_matches_ctypes_path(eng):
    from tacotron_multispeaker_b200 import torch_ops
    torch_ops.load()
    xs = [R.make_signal("sine", L, 5 + i, 16000) for i, L in enumerate([3000, 1025, 7777])]
    dense = np.zeros((3, 7777), np.float32)
    for i, x in enumerate(xs):
        dense[i, :len(x)] = x
    wav = torch.from_numpy(dense).to(eng.device)
    lengths = [len(x) for x in xs]
    for lens, so, sn in ((lengths, 16000, 20000), (None, 16000, 20000), (lengths, 44100, 16000), (lengths, 16000, 16000)):
        got = torch.ops.taco_b200.resample(eng.handle, wav, lens, so, sn)
        want = eng.resample(dense, so, sn, lengths=lens)[0]
        assert torch.equal(got, want)
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.resample(eng.handle, wav.double(), None, 16000, 20000)
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.resample(eng.handle, wav, [0, 1, 2], 16000, 20000)
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.resample(eng.handle, wav, None, 0, 20000)


def test_refusals_return_their_codes(eng):
    from tacotron_multispeaker_b200 import _abi
    x = torch.zeros(2, 1000, device=eng.device)
    y = torch.zeros(2 * 3000, device=eng.device)

    def call(so, sn, lengths=None, N=2, L=1000, L_out=1250):
        ln = None if lengths is None else np.asarray(lengths, np.int32)
        return eng.lib.taco_resample(eng._h, so, sn, C.c_void_p(x.data_ptr()), None if ln is None else ln.ctypes.data,
                                     N, L, C.c_void_p(y.data_ptr()), L_out, eng.stream)
    assert call(16000, 20000) == _abi.TACO_OK
    assert call(0, 20000) == _abi.TACO_ERR_INVALID
    assert call(16000, -20000) == _abi.TACO_ERR_INVALID
    assert call(16000, 20000, [0, 10]) == _abi.TACO_ERR_INVALID           # a length below 1
    assert call(16000, 20000, [1001, 10]) == _abi.TACO_ERR_INVALID        # a length beyond L
    assert call(16000, 20000, L_out=1249) == _abi.TACO_ERR_INVALID        # shorter than ceil(1000 * 1.25)
    assert call(16000, 20000, [799, 10], L_out=999) == _abi.TACO_OK       # ceil(799 * 1.25) = 999
    assert call(16000, 20000, N=0) == _abi.TACO_ERR_INVALID
    assert call(20000, 20000, L_out=999) == _abi.TACO_ERR_INVALID
    assert call(16000, 20000, N=2, L=1, L_out=1 << 30) == _abi.TACO_ERR_UNSUPPORTED      # N * L_out >= 2^31
    assert call(9 * 1000, 1000, L=1000, L_out=112) == _abi.TACO_ERR_UNSUPPORTED          # downsampling by more than 8
    assert call(8 * 1000, 1000, L=1000, L_out=125) == _abi.TACO_OK
    big = torch.zeros(1, (1 << 24) + 2, device=eng.device)
    yb = torch.zeros((1 << 24) + 2, device=eng.device)
    assert eng.lib.taco_resample(eng._h, 20000, 20000 * 2, C.c_void_p(big.data_ptr()), None, 1, (1 << 23) + 1,
                                 C.c_void_p(yb.data_ptr()), (1 << 24) + 2, eng.stream) == _abi.TACO_ERR_UNSUPPORTED  # > 2^24
    with pytest.raises(ValueError):
        eng.resample([np.zeros(10, np.float32), np.zeros(0, np.float32)], 16000, 20000)
    with pytest.raises(_abi.TacoError):
        eng.resample(np.zeros((2, 100), np.float32), 16000, 20000, lengths=[100, 101])
    with pytest.raises(ValueError):
        eng.resample_length(10, 16000, 0)


def _write_wav(path, pcm, rate, channels):
    with wave.open(str(path), "wb") as f:
        f.setnchannels(channels)
        f.setsampwidth(2)
        f.setframerate(rate)
        f.writeframes(np.asarray(pcm, "<i2").tobytes())


def _pcm(kind, L, channels, seed, rate):
    sig = np.stack([R.make_signal(kind, L, seed + c, rate) for c in range(channels)], axis=1)
    return np.clip(np.round(sig * 30000), -32768, 32767).astype("<i2")


def test_load_of_a_model_rate_file_equals_load_wav(eng, tmp_path):
    from tacotron_multispeaker_b200 import audio
    pcm = _pcm("chirp", 12345, 1, 4, 20000)
    _write_wav(tmp_path / "a.wav", pcm, 20000, 1)
    got = audio.load(eng, tmp_path / "a.wav", 20000)
    assert got.is_cuda and got.dtype == torch.float32
    np.testing.assert_array_equal(got.cpu().numpy(), audio.load_wav(tmp_path / "a.wav", 20000))


def test_melspectrogram_of_a_48k_stereo_file(eng, tmp_path):
    """melspectrogram(load(48 kHz stereo)) against the float64 chain: oracle resample, then the spectrogram oracle,
    within the spectrogram tests' bound."""
    from tacotron_multispeaker_b200 import audio
    pcm = np.stack([S.make_signal("chirp", 96001, 8 + c, 48000) for c in range(2)], axis=1)   # 60 Hz to 9 kHz: in band
    pcm = np.clip(np.round(pcm * 30000), -32768, 32767).astype("<i2")
    _write_wav(tmp_path / "s.wav", pcm, 48000, 2)
    y = audio.load(eng, tmp_path / "s.wav", eng.hp.sample_rate)
    assert y.shape == (R.output_length(96001, 48000, 20000),)
    lin, mel = eng.spectrogram(y)
    y64 = R.resample(R.pcm_to_float(pcm.reshape(-1), 2).astype(np.float64), 48000, 20000)
    cl, cm = S.reference_and_ratios(y64, lin.cpu().numpy(), mel.cpu().numpy(), eng.hp)
    MEASURED["48k stereo spectrogram linear"], MEASURED["48k stereo spectrogram mel"] = cl, cm
    assert cl <= S.C_BOUND and cm <= S.C_BOUND, (cl, cm)
    np.testing.assert_array_equal(audio.melspectrogram(eng, y).cpu().numpy(), mel.cpu().numpy())


def test_teacher_forced_from_a_16k_stereo_file(tmp_path):
    from tacotron_multispeaker_b200 import audio, text
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.synthesizer import Synthesizer
    text.load_symbols([chr(0x4E00 + i) for i in range(7350)])
    hp = HParams()
    syn = Synthesizer(hp).load(None, id_num=4)
    sentence = "".join(chr(0x4E00 + i) for i in (5, 17, 300, 4000, 22))
    pcm = _pcm("chirp", 4800, 2, 1, 16000)
    _write_wav(tmp_path / "rec.wav", pcm, 16000, 2)
    mel_out, align = syn.teacher_forced(sentence, 2, str(tmp_path / "rec.wav"))
    engine = syn.model._get_engine(syn.id_num)
    y = audio.load(engine, tmp_path / "rec.wav", hp.sample_rate)
    assert y.shape == (6000,)
    for wav, kw in ((y, {}), (y.cpu().numpy(), {}), (audio.read_pcm(tmp_path / "rec.wav")[0], dict(orig_sr=16000))):
        mel2, align2 = syn.teacher_forced(sentence, 2, wav, **kw)
        assert np.array_equal(mel2, mel_out) and np.array_equal(align2, align)
