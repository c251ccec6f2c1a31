"""The spectrogram analysis on the GPU (taco_spectrogram, Engine.spectrogram, the torch op, Synthesizer.teacher_forced)
against the float64 restatement of the reference's util/audio.py spectrogram / melspectrogram (tests/spectrogram_oracle.py).

Accuracy: per element, |got - want| <= (20 / ln 10) / |min_level_db| * c * sum|windowed frame| / max(1e-5, amplitude)
+ 2^-22 (mel: times the band's weight sum), with c = spectrogram_oracle.C_BOUND."""
import ctypes as C

import numpy as np
import pytest
import torch

import spectrogram_oracle as S
from oracle import audio_oracle as AO

pytestmark = pytest.mark.gpu

LENGTHS = [1, 2, 500, 1023, 1024, 1025, 5000, 20001, 250000]
MEASURED = {}   # worst c per case, printed at the end of the module


@pytest.fixture(scope="module")
def eng():
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    e = Engine(HParams(), id_num=0)       # the analysis needs no weights
    yield e
    e.close()
    if MEASURED:
        print("\nspectrogram c measured: " + ", ".join("%s %.3g" % kv for kv in sorted(MEASURED.items())))


def check_batch(e, ys, tag):
    hp = e.hp
    hop = AO.stft_parameters(hp)[1]
    lin, mel = e.spectrogram(ys)
    torch.cuda.synchronize()
    T_out = 1 + max(len(y) for y in ys) // hop
    assert lin.shape == (len(ys), T_out, hp.num_freq) and mel.shape == (len(ys), T_out, hp.num_mels)
    lin, mel = lin.cpu().numpy(), mel.cpu().numpy()
    worst_l = worst_m = 0.0
    for i, y in enumerate(ys):
        T = 1 + len(y) // hop
        cl, cm = S.reference_and_ratios(y.astype(np.float64), lin[i, :T], mel[i, :T], hp)
        worst_l, worst_m = max(worst_l, cl), max(worst_m, cm)
        assert cl <= S.C_BOUND and cm <= S.C_BOUND, (tag, len(y), cl, cm)
        # ragged batch: rows past the utterance's own frames are exact zeros (the targets' padding)
        assert not lin[i, T:].any() and not mel[i, T:].any()
    MEASURED[tag + " linear"] = worst_l
    MEASURED[tag + " mel"] = worst_m


@pytest.mark.parametrize("kind", ["silence", "sine", "noise", "chirp"])
def test_accuracy_against_float64(eng, kind):
    ys = [S.make_signal(kind, L, 10 + i) for i, L in enumerate(LENGTHS)]
    check_batch(eng, ys, kind)
    if kind == "silence":
        assert not eng.spectrogram(ys)[0].any()     # log of the 1e-5 floor is below min_level_db: exact zeros


@pytest.mark.parametrize("frame_length_ms,frame_shift_ms", [(49.95, 12.5), (50.0, 10.0), (102.4, 12.5)])
def test_other_frame_geometries(frame_length_ms, frame_shift_ms):
    # odd window (999), hop 200, and a window as long as the transform (2048, no centring offset)
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    e = Engine(HParams(frame_length_ms=frame_length_ms, frame_shift_ms=frame_shift_ms), id_num=0)
    try:
        for kind in ("noise", "chirp"):
            ys = [S.make_signal(kind, L, 40 + i) for i, L in enumerate([1, 2, 777, 5000, 20001])]
            check_batch(e, ys, "%s win %d hop %d" % (kind, AO.stft_parameters(e.hp)[2], AO.stft_parameters(e.hp)[1]))
    finally:
        e.close()


def test_batch_equals_single_calls_and_repeats(eng):
    ys = [S.make_signal("chirp", L, 70 + i) for i, L in enumerate([777, 5000, 1, 20001])]
    lin, mel = eng.spectrogram(ys)
    lin2, mel2 = eng.spectrogram(ys)
    assert torch.equal(lin, lin2) and torch.equal(mel, mel2)
    for i, y in enumerate(ys):
        l1, m1 = eng.spectrogram(y)
        T = l1.shape[0]
        assert T == eng.spectrogram_frames(len(y))
        assert torch.equal(lin[i, :T], l1) and torch.equal(mel[i, :T], m1)
    # the same batch as a dense [N, L] array with lengths
    dense = np.zeros((4, 20001), np.float32)
    for i, y in enumerate(ys):
        dense[i, :len(y)] = y
    ld, md = eng.spectrogram(dense, lengths=[len(y) for y in ys])
    assert torch.equal(ld, lin) and torch.equal(md, mel)


def test_nothing_written_outside_the_outputs(eng):
    hp = eng.hp
    ys = [S.make_signal("noise", L, 90 + i) for i, L in enumerate([5000, 1, 2345])]
    dense = np.zeros((3, 5000), np.float32)
    for i, y in enumerate(ys):
        dense[i, :len(y)] = y
    lengths = np.array([len(y) for y in ys], np.int32)
    T_out = 25                                                      # longer than the 21 frames of the longest
    want_lin, want_mel = eng.spectrogram(dense, lengths=lengths, T_out=T_out)
    wav = torch.from_numpy(dense).to(eng.device)
    G = 4096
    for which in ("both", "linear", "mel"):
        lin_buf = torch.full((2 * G + 3 * T_out * hp.num_freq,), float("nan"), device=eng.device)
        mel_buf = torch.full((2 * G + 3 * T_out * hp.num_mels,), float("nan"), device=eng.device)
        lp = C.c_void_p(lin_buf.data_ptr() + 4 * G) if which != "mel" else None
        mp = C.c_void_p(mel_buf.data_ptr() + 4 * G) if which != "linear" else None
        eng._ck(eng.lib.taco_spectrogram(eng._h, C.byref(eng.audio_params()), C.c_void_p(wav.data_ptr()), lengths.ctypes.data,
                                         3, 5000, T_out, lp, mp, eng.stream))
        torch.cuda.synchronize()
        for buf, p, want in ((lin_buf, lp, want_lin), (mel_buf, mp, want_mel)):
            if p is None:
                assert torch.isnan(buf).all()
                continue
            assert torch.isnan(buf[:G]).all() and torch.isnan(buf[-G:]).all()
            assert torch.equal(buf[G:-G].view(want.shape), want)


def test_torch_op_matches_ctypes_path(eng):
    from tacotron_multispeaker_b200 import torch_ops
    torch_ops.load()
    hp = eng.hp
    ys = [S.make_signal("sine", L, 5 + i) for i, L in enumerate([3000, 1025, 7777])]
    dense = np.zeros((3, 7777), np.float32)
    for i, y in enumerate(ys):
        dense[i, :len(y)] = y
    wav = torch.from_numpy(dense).to(eng.device)
    lengths = [len(y) for y in ys]
    args = (hp.sample_rate, hp.frame_shift_ms, hp.frame_length_ms, hp.min_level_db, hp.ref_level_db, hp.preemphasis,
            hp.num_mels, hp.num_freq)
    for lens, T_out in ((lengths, None), (None, None), (lengths, 40)):
        lin, mel = torch.ops.taco_b200.spectrogram(eng.handle, wav, lens, T_out, *args)
        want = eng.spectrogram(dense, lengths=lens, T_out=T_out)
        assert torch.equal(lin, want[0]) and torch.equal(mel, want[1])
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.spectrogram(eng.handle, wav.double(), None, None, *args)
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.spectrogram(eng.handle, wav, [0, 1, 2], None, *args)


def test_refusals_return_their_codes(eng):
    from tacotron_multispeaker_b200 import _abi
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    wav = torch.zeros(2, 1000, device=eng.device)
    out_l = torch.zeros(2 * 5 * 1025, device=eng.device)
    out_m = torch.zeros(2 * 5 * 80, device=eng.device)

    def call(e, ap, lengths, N=2, L=1000, T_out=5):
        ln = None if lengths is None else np.asarray(lengths, np.int32)
        return e.lib.taco_spectrogram(e._h, C.byref(ap), C.c_void_p(wav.data_ptr()), None if ln is None else ln.ctypes.data,
                                      N, L, T_out, C.c_void_p(out_l.data_ptr()), C.c_void_p(out_m.data_ptr()), e.stream)
    ap = eng.audio_params()
    assert call(eng, ap, None) == _abi.TACO_OK
    assert call(eng, ap, [0, 10]) == _abi.TACO_ERR_INVALID            # a length below 1
    assert call(eng, ap, [1001, 10]) == _abi.TACO_ERR_INVALID         # a length beyond L
    assert call(eng, ap, None, T_out=4) == _abi.TACO_ERR_INVALID      # T_out < 1 + 1000 // 250
    assert call(eng, ap, [249, 10], T_out=1) == _abi.TACO_OK
    assert call(eng, ap, None, N=0) == _abi.TACO_ERR_INVALID
    assert call(eng, ap, None, N=1, L=1, T_out=(1 << 31) // 1025 + 1) == _abi.TACO_ERR_UNSUPPORTED   # N T_out 1025 >= 2^31
    big = eng.audio_params()
    big.frame_length_ms = 200.0                                          # win 4000 > n_fft
    assert call(eng, big, None) == _abi.TACO_ERR_UNSUPPORTED
    e513 = Engine(HParams(num_freq=513), id_num=0)
    try:
        assert call(e513, e513.audio_params(), None) == _abi.TACO_ERR_UNSUPPORTED
    finally:
        e513.close()
    with pytest.raises(ValueError):
        eng.spectrogram([np.zeros(10, np.float32), np.zeros(0, np.float32)])
    with pytest.raises(_abi.TacoError):
        eng.spectrogram(np.zeros((2, 100), np.float32), lengths=[100, 101])


def test_teacher_forced_equals_initialize_on_the_gpu_mel(tmp_path):
    from tacotron_multispeaker_b200 import audio, text
    from tacotron_multispeaker_b200.engine import pad_targets
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.synthesizer import Synthesizer
    text.load_symbols([chr(0x4E00 + i) for i in range(7350)])
    hp = HParams()
    syn = Synthesizer(hp).load(None, id_num=4)
    sentence = "".join(chr(0x4E00 + i) for i in (5, 17, 300, 4000, 22))
    y = S.make_signal("chirp", 6000, 1)
    wav_path, png_path = tmp_path / "rec.wav", tmp_path / "align.png"
    audio.save_wav(y, str(wav_path), hp.sample_rate)
    mel_out, align = syn.teacher_forced(sentence, 2, str(wav_path), str(png_path))
    assert png_path.read_bytes()[:4] == b"\x89PNG"
    # the same run spelled out: the GPU mel of the recording, padded like the feeder's targets, through initialize
    yq = audio.load_wav(str(wav_path), hp.sample_rate)
    mel = syn.model.engine.spectrogram(yq)[1]
    targets = pad_targets([mel.cpu().numpy()], hp.outputs_per_step)
    seq = np.asarray(text.text_to_sequence2(sentence, [x.strip() for x in hp.cleaners.split(",")])[:-1], np.int32)
    syn.model.initialize(seq[None], np.asarray([seq.size], np.int32), mel_targets=targets,
                         identities=np.asarray([2], np.int32), id_num=4, teacher_force=True)
    assert np.array_equal(syn.model.mel_outputs[0].cpu().numpy(), mel_out)
    assert np.array_equal(syn.model.alignments[0].cpu().numpy(), align)
    assert mel_out.shape == (targets.shape[1], hp.num_mels) and align.shape == (seq.size, targets.shape[1])
    # an array instead of a path gives the same
    mel_out2, align2 = syn.teacher_forced(sentence, 2, yq)
    assert np.array_equal(mel_out2, mel_out) and np.array_equal(align2, align)


def test_round_trip_through_griffin_lim(eng):
    """wav -> taco_spectrogram -> taco_griffin_lim (30 iterations) -> spectrogram of the output without its first win/2
    samples (the analysis is centred, the synthesis is not): its distance to the input's spectrogram is within 5 % of the
    float64 chain's."""
    hp = eng.hp
    n_fft, hop, win = AO.stft_parameters(hp)
    L = 20000
    y = (0.6 * S.make_signal("chirp", L, 2).astype(np.float64) + 0.3 * S.make_signal("sine", L, 3)).astype(np.float32)
    T = 1 + L // hop
    lin = eng.spectrogram(y)[0]
    back = eng.griffin_lim(lin, griffin_lim_iters=30)
    lin2 = eng.spectrogram(back[win // 2:])[0]
    d_gpu = float(torch.linalg.norm(lin2[:T] - lin) / torch.linalg.norm(lin))
    lin_o = S.spectrogram_librosa(y.astype(np.float64), hp)
    back_o = AO.synthesize_wav(lin_o, hp, iters=30)
    lin2_o = S.spectrogram_librosa(back_o[win // 2:], hp)
    d_o = float(np.linalg.norm(lin2_o[:T] - lin_o) / np.linalg.norm(lin_o))
    MEASURED["round trip distance gpu"], MEASURED["round trip distance float64"] = d_gpu, d_o
    assert abs(d_gpu - d_o) <= 0.05 * d_o, (d_gpu, d_o)
