"""Every Griffin-Lim iteration of the GPU vocoder (taco_griffin_lim) and its inverse pre-emphasis, pinned step-locally against
a float64 step (``tests/griffin_lim_oracle.py``).

The waveform taco_griffin_lim returns after k iterations without inverse pre-emphasis is bit for bit the signal iteration
k + 1 frames (the kernel rebuilds each frame by adding the covering rows in the order gl_ola_kernel adds them), so iteration
k is checked by one float64 step from the kernel's own y_{k-1} against the kernel's y_k, sample by sample, with a bound
derived per sample from the operation: no error accumulates over iterations and no bound scales with the loudest sample.
The same holds for the inverse pre-emphasis: with and without it the vocoder runs the same launches, so the output without
it is exactly gl_deemph_kernel's input.

Constants, measured on a B200 at its 1000 W power limit over every case of this file:
    C_GL     = 3e-7   per-bin error of the float32 transforms, magnitudes and phase step (griffin_lim_oracle.py);
                      measured 1.3e-7 (the pure tone in one 2048-sample frame at power 2), 5.5e-8 ... 8.8e-8 for each of
                      the other geometries; largest ratio 0.58, largest median 0.075
    C_DEEMPH = 1e-5   de-emphasis error relative to lfilter(|x|); measured 3.6e-6 (a = 0.999, 250 000 samples: the carried
                      state lives 1 / (1 - a^32) = 31 warp steps), 7.1e-7 for a = 0.97
Share of (frame, bin) pairs whose phase bound caps at 2 (float32 cannot resolve those phases; CAPPED_MAX): random
spectrograms 7.4 % in one 2048-sample frame at power 2 (S spans 200 dB), at most 0.8 % elsewhere; none for the quiet,
silent and full-scale ones; 52 ... 89 % for the pure tone, whose bins at the -100 dB floor sit next to a tone 100 dB
louder (the tone's own bins keep their full bound).
"""
import ctypes as C

import numpy as np
import pytest
import torch

import griffin_lim_oracle as G

pytestmark = pytest.mark.gpu

C_GL = 3e-7
C_DEEMPH = 1e-5

# win / hop in samples at 20 kHz -> (frame_length_ms, frame_shift_ms)
GEOMETRIES = {
    "1000/250": (50.0, 12.5),    # the reference: interior frames take the four-row path
    "1000/200": (50.0, 10.0),    # generic even overlap-add
    "999/250": (49.95, 12.5),    # odd window: scalar loads and stores
    "2048/125": (102.4, 6.25),   # the whole transform, 17 overlapping frames
    "600/250": (30.0, 12.5),
    "200/250": (10.0, 12.5),     # hop > win: gaps between frames, no overlap
}
CHECKPOINTS = (0, 1, 2, 7, 31)   # iteration k is the step y_{k-1} -> y_k; 0 is the zero-phase start
POWERS = (1.5, 1.0, 2.0)
# share of (frame, bin) pairs whose phase bound hits its cap of 2 (the float32 transform cannot resolve the bin's phase)
CAPPED_MAX = {"random": 0.1, "quiet": 0.01, "silence": 0.0, "full": 0.0, "tone": 0.95}
MEDIAN_MAX = 0.25


@pytest.fixture(scope="module")
def engines():
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    cache = {}

    def get(frame_length_ms, frame_shift_ms):
        key = (frame_length_ms, frame_shift_ms)
        if key not in cache:
            cache[key] = Engine(HParams(frame_length_ms=frame_length_ms, frame_shift_ms=frame_shift_ms), id_num=0)
        return cache[key]
    yield get
    for e in cache.values():
        e.close()


def spectrogram(T, seed, lo=-0.1, hi=1.05):
    rng = np.random.default_rng(seed)
    # smooth-ish in time and frequency, leaving [0, 1] at both ends so that the clip is exercised
    x = rng.uniform(lo, hi, (T, 1025)).astype(np.float32)
    x[:, 1:] = 0.5 * (x[:, 1:] + x[:, :-1])
    return x


@pytest.fixture(scope="module")
def tone(engines):
    """taco_spectrogram of a 440 Hz sine at half scale, 1000 frames: a few loud bins, the rest at the -100 dB floor."""
    eng = engines(*GEOMETRIES["1000/250"])
    wav = (0.5 * np.sin(2 * np.pi * 440.0 * np.arange(999 * 250) / 20000.0)).astype(np.float32)
    lin, _ = eng.spectrogram(wav, T_out=1000)
    return lin.cpu().numpy()


def inputs(T, seed, tone):
    return {
        "random": spectrogram(T, seed),
        "quiet": spectrogram(T, seed + 1, lo=0.0, hi=0.3),     # -80 ... -50 dB: every |X| below 1e-4
        "silence": np.zeros((T, 1025), np.float32),
        "full": np.ones((T, 1025), np.float32),
        "tone": tone[:T],
    }


def hparams(eng, power):
    hp = eng.hp.copy()
    hp.power = power
    return hp


def vocode(eng, lin, iters, power=None, preemphasis=0.0, T=None, batch_stride=0):
    """taco_griffin_lim on a device batch lin [N, >= T, 1025]: wav [N, L] on the host (float32)."""
    N = lin.shape[0]
    T = lin.shape[1] if T is None else T
    ap = eng.audio_params(iters)
    ap.preemphasis = preemphasis
    if power is not None:
        ap.power = power
    L = eng.lib.taco_wav_length(C.byref(ap), T)
    out = torch.empty(N, L, device=eng.device)
    eng._ck(eng.lib.taco_griffin_lim(eng._h, C.byref(ap), C.c_void_p(lin.data_ptr()), N, T, batch_stride,
                                     C.c_void_p(out.data_ptr()), eng.stream))
    return out.cpu().numpy()


def check_steps(hp, S, names, wavs, ks, tag):
    """Step-local check of iterations ks of every utterance; prints one line per utterance and asserts after printing."""
    failures = []
    for n, name in enumerate(names):
        rs = [G.gl_local_check(None if k == 0 else wavs[k - 1][n], wavs[k][n], S[n], hp, C_GL) for k in ks]
        worst = max(rs, key=lambda r: r.max_ratio)
        print("%s %-7s max ratio %.3g  median %.3g  capped %.4f  needs c %.3g" % (
            tag, name, worst.max_ratio, max(r.median_ratio for r in rs), max(r.capped for r in rs),
            max(r.needed_c for r in rs)))
        for k, r in zip(ks, rs):
            if not (r.max_ratio <= 1.0 and r.median_ratio <= MEDIAN_MAX and r.capped <= CAPPED_MAX[name]):
                failures.append("%s %s k=%d: %s" % (tag, name, k, r))
    assert not failures, "\n".join(failures)


@pytest.mark.parametrize("T", [1, 2, 3, 6, 7, 24])
@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_iterations_are_float64_steps(engines, tone, geom, T):
    """Checkpoints 0, 1, 2, 7, 31 of five spectrograms (the clip, a quiet passage, silence, full scale and a pure tone's
    near-zero bins) at each power, every frame geometry and frame counts where every frame is an edge frame (T <= 6), the
    first interior frame (T = 7) and beyond."""
    eng = engines(*GEOMETRIES[geom])
    ins = inputs(T, 10 * T + len(geom), tone)
    names = list(ins)
    lin_host = np.stack([ins[k] for k in names])
    lin = torch.from_numpy(lin_host).to(eng.device)
    calls = sorted({0} | {k for c in CHECKPOINTS if c for k in (c - 1, c)})
    for power in POWERS:
        hp = hparams(eng, power)
        wavs = {k: vocode(eng, lin, k, power) for k in calls}
        check_steps(hp, G.mags64(lin_host, hp), names, wavs, CHECKPOINTS,
                    "%s T=%d p=%.1f" % (geom, T, power))


def test_last_iteration_at_full_size(engines):
    """Iteration 100 (the hparams default's last) of a batch of 32 utterances of 1000 frames at the reference geometry."""
    eng = engines(*GEOMETRIES["1000/250"])
    lin_host = np.stack([spectrogram(1000, 500 + i) for i in range(32)])
    lin = torch.from_numpy(lin_host).to(eng.device)
    wavs = {k: vocode(eng, lin, k) for k in (99, 100)}
    check_steps(eng.hp, G.mags64(lin_host, eng.hp), ["random"] * 32, wavs, (100,), "1000/250 T=1000 N=32")


def test_strided_batch(engines):
    """33 utterances of 24 frames read from rows of 30 frames (the rows past 24 hold NaN and must not be read), iteration 5."""
    eng = engines(*GEOMETRIES["1000/250"])
    lin_host = np.stack([spectrogram(24, 900 + i) for i in range(33)])
    big = torch.full((33, 30, 1025), float("nan"), device=eng.device)
    big[:, :24] = torch.from_numpy(lin_host).to(eng.device)
    wavs = {k: vocode(eng, big, k, T=24, batch_stride=30 * 1025) for k in (4, 5)}
    check_steps(eng.hp, G.mags64(lin_host, eng.hp), ["random"] * 33, wavs, (5,), "1000/250 T=24 N=33 strided")


# (frame_length_ms, frame_shift_ms, T): L = (T - 1) hop + win samples
DEEMPH_LENGTHS = {
    20: (1.0, 0.5, 1),            # shorter than one warp step
    1024: (51.2, 12.5, 1),        # segments of 32: one step per warp
    1025: (51.25, 12.5, 1),       # segments of 64: warp 16 holds one sample, warps 17-31 none
    250000: (50.0, 12.5, 997),
}


@pytest.mark.parametrize("L", list(DEEMPH_LENGTHS))
@pytest.mark.parametrize("a", [0.97, 0.999, 0.5])
def test_inverse_preemphasis_is_lfilter_of_its_input(engines, a, L):
    fl, fs, T = DEEMPH_LENGTHS[L]
    eng = engines(fl, fs)
    lin = torch.from_numpy(np.stack([spectrogram(T, L), spectrogram(T, L + 1, lo=0.0, hi=0.3)])).to(eng.device)
    x = vocode(eng, lin, 1)
    got = vocode(eng, lin, 1, preemphasis=a)
    assert x.shape == got.shape == (2, L)
    for n in range(2):
        q, i, need = G.deemph_check(got[n], x[n], a, C_DEEMPH)
        print("deemph a=%g L=%d utterance %d: max ratio %.3g at %d, needs c %.3g" % (a, L, n, q, i, need))
        assert q <= 1.0, (a, L, n, q, i)


def test_zero_preemphasis_launches_nothing(engines):
    eng = engines(*GEOMETRIES["1000/250"])
    lin = torch.from_numpy(spectrogram(9, 3)).to(eng.device)
    plain = eng.griffin_lim(lin, 2, inv_preemphasis=False)
    counts = []
    for a in (0.0, 0.97):
        ap = eng.audio_params(2)
        ap.preemphasis = a
        out = torch.empty_like(plain)
        c0 = eng.launch_count()
        eng._ck(eng.lib.taco_griffin_lim(eng._h, C.byref(ap), C.c_void_p(lin.data_ptr()), 1, 9, 0,
                                         C.c_void_p(out.data_ptr()), eng.stream))
        counts.append(eng.launch_count() - c0)
        if a == 0.0:
            assert torch.equal(out, plain)
        else:
            assert not torch.equal(out, plain)
    assert counts == [4 + 2, 4 + 2 + 1], counts
