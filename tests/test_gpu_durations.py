"""Per-symbol durations on the GPU (taco_durations, Engine.durations, the torch op, Synthesizer.align) against the float64
restatement of Glow-TTS's monotonic alignment search (tests/alignment_oracle.py).

Where the optimum is unique by construction (uniform matrices: every path ties and the tie rule decides; planted paths)
the durations equal the oracle's exactly.  On random and decoder alignments CUDA's double log may differ from numpy's in
the last bit, so a near-tie may flip: there the GPU path must be a valid path whose float64 score is within
1e-9 (1 + |opt|) of the oracle's optimum."""
import ctypes as C
import wave

import numpy as np
import pytest
import torch

import alignment_oracle as A

pytestmark = pytest.mark.gpu

# (N, T_in, steps, r): batch sizes 1 / 7 / 70, T_in at the warp edges and the 512 cap, Y from X up to 2000
EXACT_CASES = [(1, 1, 2000, 1), (7, 2, 300, 5), (70, 31, 400, 1), (7, 32, 2000, 5), (1, 32, 32, 1), (70, 33, 120, 5),
               (7, 511, 2000, 1), (1, 512, 512, 5), (7, 512, 2000, 5), (70, 512, 600, 1)]
DIFFERING = {}   # paths that differ from the oracle's (legitimate near-ties), printed at the end of the module


@pytest.fixture(scope="module")
def engines():
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    es = {r: Engine(HParams(outputs_per_step=r), id_num=0) for r in (1, 5)}   # durations need no weights
    yield es
    for e in es.values():
        e.close()
    if DIFFERING:
        print("\ndurations: paths differing from the oracle's: " + ", ".join("%s %d/%d" % (k, v[0], v[1])
                                                                          for k, v in sorted(DIFFERING.items())))


def geometry(rng, N, T_in, steps, r):
    """Text lengths and frame counts for a batch: the longest text, one symbol, Y == X, Y == steps, every F % r."""
    X = rng.integers(1, T_in + 1, N)
    X[0] = T_in
    if N > 1:
        X[1] = 1
    Y = np.asarray([rng.integers(x, steps + 1) for x in X])
    Y[0] = steps if N == 1 else T_in
    if N > 2:
        Y[2] = steps
    F = Y * r - np.arange(N) % r                             # ceil(F / r) == Y
    return X.astype(np.int32), F.astype(np.int32)


def make_batch(rng, N, T_in, steps, r, kind):
    """(a [N, T_in, steps] float32, X, F, expected durations [N, T_in]).  Cells outside rows < X, columns < Y hold
    unrelated values."""
    X, F = geometry(rng, N, T_in, steps, r)
    a = rng.random((N, T_in, steps), dtype=np.float32)
    want = np.zeros((N, T_in), np.int32)
    for n in range(N):
        x, f = int(X[n]), int(F[n])
        y = A.steps_for(f, r)
        if kind == "uniform":
            a[n, :x, :y] = 1.0 / x
            want[n, :x] = [r] * (x - 1) + [f - (x - 1) * r]
        else:
            p = A.planted_path(rng, x, y)
            a[n, :x, :y] = 1e-3
            a[n, p, np.arange(y)] = 0.9
            want[n] = A.durations_of_path(p, f, r, T_in)
    return a, X, F, want


def gpu(eng, a, X, F):
    return eng.durations(torch.from_numpy(a).to(eng.device), X, F).cpu().numpy()


@pytest.mark.parametrize("N,T_in,steps,r", EXACT_CASES)
@pytest.mark.parametrize("kind", ["uniform", "planted"])
def test_exact_on_unique_optima(engines, N, T_in, steps, r, kind):
    rng = np.random.default_rng(N * 1000 + T_in + steps + r)
    a, X, F, want = make_batch(rng, N, T_in, steps, r, kind)
    got = gpu(engines[r], a, X, F)
    assert got.dtype == np.int32 and got.shape == (N, T_in)
    for n in range(N):
        oracle = A.durations(a[n], int(X[n]), int(F[n]), r)[0]
        assert np.array_equal(oracle, want[n]), n
        assert np.array_equal(got[n], want[n]), (n, X[n], F[n])


def check_optimal(tag, a, X, F, r, got):
    """The GPU durations form a path in the band whose float64 score is the optimum's to 1e-9 (1 + |opt|)."""
    differ = 0
    for n in range(len(X)):
        x, f = int(X[n]), int(F[n])
        d_ref, p_ref, Q = A.durations(a[n], x, f, r)
        path = A.path_from_durations(got[n], x, f, r)      # asserts monotonic, in the band, sum F, each >= 1
        s = A.scores(a[n], x, A.steps_for(f, r))
        opt = Q[-1, x - 1]
        assert abs(A.path_score(s, path) - opt) <= 1e-9 * (1 + abs(opt)), (tag, n)
        differ += not np.array_equal(path, p_ref)
    d = DIFFERING.setdefault(tag, [0, 0])
    d[0] += differ
    d[1] += len(X)


def column_softmax(rng, N, T_in, steps, sharp):
    z = rng.normal(0.0, sharp, (N, T_in, steps))
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return (e / e.sum(axis=1, keepdims=True)).astype(np.float32)


@pytest.mark.parametrize("N,T_in,steps,r", [(7, 33, 500, 1), (70, 100, 200, 5), (7, 512, 2000, 1), (32, 64, 1000, 5)])
@pytest.mark.parametrize("sharp", [0.5, 4.0])
def test_optimal_on_random_column_softmax(engines, N, T_in, steps, r, sharp):
    rng = np.random.default_rng(T_in + steps)
    a = column_softmax(rng, N, T_in, steps, sharp)
    X, F = geometry(rng, N, T_in, steps, r)
    check_optimal("softmax", a, X, F, r, gpu(engines[r], a, X, F))


def test_optimal_on_decoder_alignments():
    """Teacher-forced attention of a random-init model (config-3 shapes, r = 5): batch 16, T_in 100, 1000 frames."""
    from conftest import make_inputs
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    e = Engine(hp, id_num=0)
    e.load_weights(random_init(hp, 0, seed=21))
    ids, lengths, _ = make_inputs(16, 100, 0, seed=3)
    rng = np.random.default_rng(4)
    targets = rng.random((16, 1000, hp.num_mels), dtype=np.float32)
    _, _, al, steps = e.forward(ids, lengths, None, targets, teacher_force=True, want_linear=False)
    assert steps == 200
    F = np.asarray([rng.integers(5 * int(x), 1001) for x in lengths], np.int32)
    F[0] = 1000
    got = e.durations(al, lengths, F).cpu().numpy()
    check_optimal("decoder", al.cpu().numpy(), lengths, F, 5, got)
    e.close()


def test_padding_is_never_read_and_nothing_outside_is_written(engines):
    eng = engines[5]
    rng = np.random.default_rng(8)
    N, T_in, steps = 7, 70, 300
    a, X, F, _ = make_batch(rng, N, T_in, steps, 5, "planted")
    a = column_softmax(rng, N, T_in, steps, 2.0) * 0.5 + a * 0.5
    want = gpu(eng, a, X, F)
    b = a.copy()
    for n in range(N):
        b[n, X[n]:] = np.nan
        b[n, :, A.steps_for(F[n], 5):] = np.nan
    assert np.array_equal(gpu(eng, b, X, F), want)
    for n in range(N):
        assert not want[n, X[n]:].any() and (want[n, :X[n]] >= 1).all() and want[n].sum() == F[n]
    G = 4096
    buf = torch.full((2 * G + N * T_in,), -12345, dtype=torch.int32, device=eng.device)
    a_dev = torch.from_numpy(b).to(eng.device)
    eng._ck(eng.lib.taco_durations(eng._h, C.c_void_p(a_dev.data_ptr()), N, T_in, steps, X.ctypes.data, F.ctypes.data,
                                   C.c_void_p(buf.data_ptr() + 4 * G), eng.stream))
    torch.cuda.synchronize()
    buf = buf.cpu().numpy()
    assert (buf[:G] == -12345).all() and (buf[-G:] == -12345).all()
    assert np.array_equal(buf[G:-G].reshape(N, T_in), want)


def test_batch_equals_single_calls_and_repeats(engines):
    eng = engines[1]
    rng = np.random.default_rng(9)
    N, T_in, steps = 9, 200, 700
    a = column_softmax(rng, N, T_in, steps, 3.0)
    X, F = geometry(rng, N, T_in, steps, 1)
    a_dev = torch.from_numpy(a).to(eng.device)
    first = eng.durations(a_dev, X, F)
    for _ in range(3):
        assert torch.equal(eng.durations(a_dev, X, F), first)
    for n in range(N):
        assert torch.equal(eng.durations(a_dev[n:n + 1], X[n:n + 1], F[n:n + 1]), first[n:n + 1])


def test_refusals_return_their_codes(engines):
    from tacotron_multispeaker_b200 import _abi
    eng = engines[5]
    a = torch.zeros(2, 8, 10, device=eng.device)
    out = torch.zeros(2 * 8, dtype=torch.int32, device=eng.device)

    def call(lens=(8, 3), frames=(50, 20), N=2, T_in=8, steps=10, align=True, lens_ptr=True, frames_ptr=True, out_ptr=True):
        ln, fr = np.asarray(lens, np.int32), np.asarray(frames, np.int32)
        return eng.lib.taco_durations(eng._h, C.c_void_p(a.data_ptr()) if align else None, N, T_in, steps,
                                      ln.ctypes.data if lens_ptr else None, fr.ctypes.data if frames_ptr else None,
                                      C.c_void_p(out.data_ptr()) if out_ptr else None, eng.stream)
    assert call() == _abi.TACO_OK
    assert call(align=False) == _abi.TACO_ERR_INVALID
    assert call(lens_ptr=False) == _abi.TACO_ERR_INVALID
    assert call(frames_ptr=False) == _abi.TACO_ERR_INVALID
    assert call(out_ptr=False) == _abi.TACO_ERR_INVALID
    assert call(N=0) == _abi.TACO_ERR_INVALID
    assert call(steps=0) == _abi.TACO_ERR_INVALID
    assert call(lens=(0, 3)) == _abi.TACO_ERR_INVALID                  # a text length below 1
    assert call(lens=(9, 3)) == _abi.TACO_ERR_INVALID                  # beyond T_in
    assert call(frames=(0, 20)) == _abi.TACO_ERR_INVALID
    assert call(frames=(51, 20)) == _abi.TACO_ERR_INVALID              # beyond steps * r
    assert call(frames=(35, 20)) == _abi.TACO_ERR_INVALID              # 7 steps for 8 symbols: no path
    assert call(frames=(50, 10)) == _abi.TACO_ERR_INVALID              # 2 steps for 3
    assert call(frames=(36, 11)) == _abi.TACO_OK                       # ceil(36 / 5) = 8 and ceil(11 / 5) = 3 steps
    assert call(T_in=513, lens=(8, 3)) == _abi.TACO_ERR_UNSUPPORTED
    assert call(steps=65537) == _abi.TACO_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        eng.durations(a, [8], [50, 20])
    with pytest.raises(_abi.TacoError):
        eng.durations(a, [8, 3], [50, 10])


def test_torch_op_matches_ctypes_path(engines):
    from tacotron_multispeaker_b200 import torch_ops
    torch_ops.load()
    eng = engines[5]
    rng = np.random.default_rng(12)
    a = column_softmax(rng, 5, 40, 150, 2.0)
    X, F = geometry(rng, 5, 40, 150, 5)
    a_dev = torch.from_numpy(a).to(eng.device)
    got = torch.ops.taco_b200.durations(eng.handle, a_dev, X.tolist(), F.tolist())
    assert got.dtype == torch.int32 and torch.equal(got, eng.durations(a_dev, X, F))
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.durations(eng.handle, a_dev.double(), X.tolist(), F.tolist())
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.durations(eng.handle, a_dev, X.tolist()[:4], F.tolist())
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.durations(eng.handle, a_dev, [41] + X.tolist()[1:], F.tolist())
    with pytest.raises(RuntimeError):
        torch.ops.taco_b200.durations(eng.handle, a_dev, X.tolist(), [5 * 150 + 1] + F.tolist()[1:])


# ---- Synthesizer.align ------------------------------------------------------------------------------------------------

def _write_wav(path, sig, rate, channels):
    rng = np.random.default_rng(len(sig))
    pcm = np.stack([sig * (0.9 + 0.1 * c) + 0.01 * rng.normal(size=sig.size) for c in range(channels)], axis=1)
    with wave.open(str(path), "wb") as f:
        f.setnchannels(channels)
        f.setsampwidth(2)
        f.setframerate(rate)
        f.writeframes(np.clip(np.round(pcm * 20000), -32768, 32767).astype("<i2").tobytes())


def _chirp(L, rate, seed):
    t = np.arange(L) / rate
    return (0.5 * np.sin(2 * np.pi * (150 + 900 * t + 50 * seed) * t)).astype(np.float32)


@pytest.fixture(scope="module")
def syn():
    from tacotron_multispeaker_b200 import text
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.synthesizer import Synthesizer
    text.load_symbols([chr(0x4E00 + i) for i in range(7350)])
    return Synthesizer(HParams()).load(None, id_num=4)


def sentence(*ids):
    return "".join(chr(0x4E00 + i) for i in ids)


def test_align_of_one_utterance_equals_teacher_forced(syn, tmp_path):
    _write_wav(tmp_path / "one.wav", _chirp(9000, 16000, 1), 16000, 2)
    t = sentence(5, 17, 300, 4000, 22, 9, 81)
    (d, al), = syn.align([t], [2], [tmp_path / "one.wav"])
    _, al_tf = syn.teacher_forced(t, 2, str(tmp_path / "one.wav"))
    F = 1 + 11250 // 250                                        # 9000 samples at 16 kHz -> 11250 at 20 kHz
    assert al.dtype == np.float32 and al.shape == (7, F) and d.dtype == np.int32 and d.shape == (7,)
    assert np.array_equal(al, al_tf[:, :F])
    check_optimal("align", al[None], np.int32([7]), np.int32([F]), 1, d[None])


def test_ragged_batch_equals_the_run_spelled_out(syn, tmp_path):
    from tacotron_multispeaker_b200 import audio
    from tacotron_multispeaker_b200.engine import pad_inputs
    from tacotron_multispeaker_b200.text import text_to_sequence2
    _write_wav(tmp_path / "s16.wav", _chirp(6400, 16000, 0), 16000, 2)
    _write_wav(tmp_path / "m20.wav", _chirp(12345, 20000, 1), 20000, 1)
    _write_wav(tmp_path / "m48.wav", _chirp(30000, 48000, 2), 48000, 1)
    arr = _chirp(4000, 16000, 3)
    ten = torch.from_numpy(_chirp(11111, 16000, 4)).cuda()
    texts = [sentence(1, 2, 3, 4, 5), sentence(*range(100, 130)), sentence(7, 8), sentence(*range(200, 215)),
             sentence(*range(300, 312))]
    wavs = [tmp_path / "s16.wav", str(tmp_path / "m20.wav"), tmp_path / "m48.wav", arr, ten]
    ids = [0, 3, 1, 2, 3]
    got = syn.align(texts, ids, wavs, orig_sr=16000)

    engine = syn.model._get_engine(syn.id_num)
    ys = [audio.load(engine, w, 20000) for w in wavs[:3]] + [audio.resample(engine, torch.as_tensor(w), 16000, 20000)
                                                           for w in wavs[3:]]
    frames = [engine.spectrogram_frames(y.numel()) for y in ys]
    T = max(frames) + 1                                         # pad_targets' length at r = 1
    _, mel = engine.spectrogram(ys, T_out=T)
    seqs = [text_to_sequence2(t)[:-1] for t in texts]
    lengths = np.int32([len(s) for s in seqs])
    _, _, al, _ = engine.forward(pad_inputs(seqs), lengths, np.int32(ids), mel, teacher_force=True, want_linear=False)
    d = engine.durations(al, lengths, frames).cpu().numpy()
    al = al.cpu().numpy()
    assert len(got) == 5
    for n, (dn, an) in enumerate(got):
        assert np.array_equal(dn, d[n, :lengths[n]]) and np.array_equal(an, al[n, :lengths[n], :frames[n]]), n
        assert dn.sum() == frames[n]
    check_optimal("align", al, lengths, np.int32(frames), 1, d)


def test_align_raises_for_each_bad_utterance(syn):
    good = _chirp(8000, 20000, 0)
    with pytest.raises(ValueError, match="utterance 1:.*513 symbols"):
        syn.align([sentence(1, 2), sentence(*range(513))], [0, 0], [good, good])
    with pytest.raises(ValueError, match="utterance 1:.*max_iters.*400"):
        syn.align([sentence(1, 2), sentence(3)], [0, 0], [good, np.zeros(100000, np.float32)])   # 401 frames
    with pytest.raises(ValueError, match="utterance 0:.*5 decoder steps for 6 symbols"):
        syn.align([sentence(*range(6)), sentence(3)], [0, 0], [np.zeros(1000, np.float32), good])
    with pytest.raises(ValueError):
        syn.align([sentence(1)], [0, 1], [good])
