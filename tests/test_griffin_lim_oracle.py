"""The float64 Griffin-Lim step of ``tests/griffin_lim_oracle.py`` against the oracle's whole-run restatement, and the teeth of
its step-local check and of the inverse pre-emphasis check: each planted defect must fail by a wide margin.  No GPU."""
import numpy as np
import pytest
from scipy.signal import lfilter

import griffin_lim_oracle as G
from oracle import audio_oracle as A
from tacotron_multispeaker_b200.hparams import HParams

C = 1e-7   # an FFT error of the size the GPU tests use
GEOMETRIES = {"1000/250": (50.0, 12.5), "999/200": (49.95, 10.0)}


def spectrogram(T, seed, lo=-0.1, hi=1.05):
    rng = np.random.default_rng(seed)
    x = rng.uniform(lo, hi, (T, 1025)).astype(np.float32)
    x[:, 1:] = 0.5 * (x[:, 1:] + x[:, :-1])
    return x


def trajectory(S, hp, k):
    y = G.gl_start64(S, hp).y
    for _ in range(k):
        y = G.gl_step64(y, S, hp).y
    return y


@pytest.mark.parametrize("geom", list(GEOMETRIES))
@pytest.mark.parametrize("k", [0, 1, 3])
def test_composed_steps_equal_the_oracle(geom, k):
    hp = HParams(frame_length_ms=GEOMETRIES[geom][0], frame_shift_ms=GEOMETRIES[geom][1])
    S = G.mags64(spectrogram(9, 5 + k), hp)
    got = trajectory(S, hp, k)
    want = A.griffin_lim_tf(S, hp, iters=k)
    assert got.shape == want.shape
    assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))


def test_mags64_is_the_oracles_magnitude():
    hp = HParams(power=2.0)
    x = spectrogram(3, 1)
    want = np.power(A.db_to_amp(A.denormalize(x.astype(np.float64), hp) + hp.ref_level_db), 2.0)
    assert np.array_equal(G.mags64(x, hp), want)
    assert G.mags64(np.zeros((1, 1025), np.float32), hp)[0, 0] == pytest.approx(1e-8)    # -80 dB, squared


@pytest.fixture(scope="module")
def case():
    hp = HParams()
    S = G.mags64(spectrogram(11, 42), hp)
    y2 = trajectory(S, hp, 2)
    return hp, S, y2, G.gl_step64(y2, S, hp).y


def test_exact_trajectory_passes_at_c_zero(case):
    hp, S, y2, y3 = case
    for yk, yk1 in ((None, G.gl_start64(S, hp).y), (y2, y3)):
        r = G.gl_local_check(yk, yk1, S, hp, 0.0)
        assert r.max_ratio <= 1.0 and r.needed_c == 0.0, r


def test_one_sample_at_ten_times_its_bound_fails(case):
    hp, S, y2, y3 = case
    st = G.gl_step64(y2, S, hp)
    bad = y3.copy()
    m = len(bad) // 3
    bad[m] += 10.0 * G.gl_local_bound(st, C)[m]
    r = G.gl_local_check(y2, bad, S, hp, C)
    assert r.max_ratio > 9.0 and r.worst[0] == m, r


def test_nan_fails(case):
    hp, S, y2, y3 = case
    bad = y3.copy()
    bad[17] = np.nan
    r = G.gl_local_check(y2, bad, S, hp, C)
    assert r.max_ratio == np.inf and r.needed_c == np.inf, r


def test_c_ten_times_tighter_than_a_planted_perturbation_fails(case):
    hp, S, y2, y3 = case
    st = G.gl_step64(y2, S, hp)
    sign = np.where(np.random.default_rng(3).random(len(y3)) < 0.5, -1.0, 1.0)
    bad = y3 + sign * G.gl_local_bound(st, C)
    assert G.gl_local_check(y2, bad, S, hp, C, search=False).max_ratio <= 1.0 + 1e-9
    r = G.gl_local_check(y2, bad, S, hp, C / 10)
    # the final roundings' part of the bound does not scale with c: the ratio grows less than 10x, but the search finds the
    # planted c
    assert r.max_ratio > 5.0 and 0.9 * C < r.needed_c < 1.1 * C, r


def _defective_step(y, S, hp, *, window=None, drop_last=False, offset=0):
    """gl_step64 with one defect: another window, the last frame left out of the overlap-add, frames read `offset` samples
    late."""
    win, hop = G.geometry(hp)
    T = S.shape[0]
    w = A.hann_periodic(win) if window is None else window
    yp = np.concatenate([np.asarray(y, np.float64), np.zeros(offset)])[offset:]
    idx = np.arange(T)[:, None] * hop + np.arange(win)[None, :]
    X = np.fft.rfft(yp[idx] * w, G.N_FFT, axis=-1)
    r = np.fft.irfft(S * X / np.maximum(1e-8, np.abs(X)), G.N_FFT, axis=-1)[:, :win] * w
    out = np.zeros(len(y))
    for t in range(T - 1 if drop_last else T):
        out[t * hop:t * hop + win] += r[t]
    return out


@pytest.mark.parametrize("defect", ["symmetric_hann", "drop_last_frame", "frame_offset", "no_power"])
def test_defective_steps_fail_by_a_wide_margin(case, defect):
    hp, S, y2, _ = case
    win, _ = G.geometry(hp)
    if defect == "symmetric_hann":
        got = _defective_step(y2, S, hp, window=0.5 - 0.5 * np.cos(2 * np.pi * np.arange(win) / (win - 1)))
    elif defect == "drop_last_frame":
        got = _defective_step(y2, S, hp, drop_last=True)
    elif defect == "frame_offset":
        got = _defective_step(y2, S, hp, offset=1)
    else:
        got = _defective_step(y2, S ** (1.0 / hp.power), hp)
    assert np.max(np.abs(got - G.gl_step64(y2, S, hp).y)) > 0       # the defect changes the output
    r = G.gl_local_check(y2, got, S, hp, C)
    assert r.max_ratio > 100.0, (defect, r)


def test_zero_phase_start_without_power_fails():
    hp = HParams()
    x = spectrogram(5, 8)
    S = G.mags64(x, hp)
    got = G.gl_start64(S ** (1.0 / hp.power), hp).y
    assert G.gl_local_check(None, got, S, hp, C).max_ratio > 100.0


def segmented_scan(x, a, carry_factor=None, restart=False):
    """gl_deemph_kernel's scan in float64: 32 segments of seg samples (seg: ceil(L / 32) rounded up to 32), each filtered
    on its own, the segment end states chained with factor a^seg (carry_factor(a, seg) to plant a defect) and
    carry * a^(k+1) added to sample k of each segment.  restart: no carry between segments."""
    x = np.asarray(x, np.float64)
    L = len(x)
    seg = (((L + 31) // 32) + 31) & ~31
    f = a ** seg if carry_factor is None else carry_factor(a, seg)
    z = np.zeros(L)
    cc = 0.0
    for w in range(32):
        s, e = min(L, w * seg), min(L, w * seg + seg)
        local = lfilter([1.0], [1.0, -a], x[s:e])
        carry = 0.0 if restart else cc
        z[s:e] = local + carry * a ** np.arange(1, e - s + 1)
        cc = f * cc + (local[-1] if e > s else 0.0)
    return z


@pytest.mark.parametrize("L", [20, 1025, 250000])
@pytest.mark.parametrize("a", [0.97, 0.999, 0.5])
def test_deemph_check_accepts_the_segmented_scan(L, a):
    x = np.random.default_rng(L).standard_normal(L)
    q, _, _ = G.deemph_check(segmented_scan(x, a), x, a, 1e-12)
    assert q <= 1.0, q


@pytest.mark.parametrize("a", [0.97, 0.999])
@pytest.mark.parametrize("defect", ["restart", "a^(seg-1)"])
def test_deemph_check_rejects_a_broken_carry(a, defect):
    L = 1025                       # seg = 64: samples past the first segment depend on the carries
    x = np.random.default_rng(1).standard_normal(L)
    if defect == "restart":
        got = segmented_scan(x, a, restart=True)
    else:
        got = segmented_scan(x, a, carry_factor=lambda a, seg: a ** (seg - 1))
    q, i, _ = G.deemph_check(got, x, a, 1e-5)     # the c of the GPU tests
    assert q > 20.0 and i >= 64, (q, i)
