"""float64 restatement of librosa 0.5.1 ``core.resample`` / ``core.load`` with resampy 0.1.5's ``kaiser_best`` filter, for
the tests.  Neither library is installed: the conventions below are restated from memory of those releases and stay
unpinned against them.  Each has a test of its own in ``tests/test_resample_oracle.py``.

* Filter: ``interp_win = kaiser(2 n + 1, beta)[n:] * rolloff * sinc(rolloff * linspace(0, 64, n + 1))`` with
  ``n = 64 * 512`` (32 769 entries), times ``ratio`` when ``ratio = sr_new / sr_orig < 1``;
  ``interp_delta[:-1] = diff(interp_win)``, last entry 0.
* ``resample_f``: ``scale = min(1, ratio)``, ``index_step = int(scale * 512)`` (truncated); a double time register
  advanced by ``1 / ratio`` per output; output ``t`` takes ``n = int(register)`` and, from ``frac = scale * (register - n)``,
  a left wing of ``min(n + 1, (nwin - offset) // index_step)`` taps and, from ``scale - frac``, a right wing of
  ``min(L - n - 1, ...)`` taps, each weight ``interp_win[o] + eta * interp_delta[o]``.  Samples outside ``[0, L)``
  contribute nothing.  ``int(L * ratio)`` outputs.
* librosa: equal rates return the input; otherwise ``fix_length`` zero-pads to ``ceil(L * ratio)``.  ``load`` converts int16
  as ``float32(pcm) * (1 / 32768)`` and mixes channels with ``np.mean`` in float32.

The keyword switches (``exact_positions``, ``exact_step``, ``length``) restate deliberate mistakes; the tests use them to
show that each mistake would be caught.
"""
from __future__ import annotations

import math

import numpy as np
import scipy.signal

NUM_ZEROS = 64
PRECISION = 9
NUM_TABLE = 1 << PRECISION                     # table entries per zero crossing
BETA = 14.769656459379492
ROLLOFF = 0.9475937167399596


def filter_table():
    """resampy's kaiser_best ``half_window`` (32 769 entries)."""
    n = NUM_TABLE * NUM_ZEROS
    sinc_win = ROLLOFF * np.sinc(ROLLOFF * np.linspace(0, NUM_ZEROS, num=n + 1, endpoint=True))
    taper = scipy.signal.windows.kaiser(2 * n + 1, BETA)[n:]
    return taper * sinc_win


def tables(sr_orig, sr_new):
    """(interp_win, interp_delta) as resample() hands them to resample_f."""
    ratio = float(sr_new) / sr_orig
    win = filter_table()
    if ratio < 1:
        win = win * ratio
    delta = np.zeros_like(win)
    delta[:-1] = np.diff(win)
    return win, delta


def index_step(sr_orig, sr_new, exact_step=False):
    scale = min(1.0, float(sr_new) / sr_orig)
    return scale * NUM_TABLE if exact_step else int(scale * NUM_TABLE)


def positions(sr_orig, sr_new, count, exact_positions=False):
    """Per output t < count: (n, offset_l, eta_l, offset_r, eta_r) of resample_f, eta in float64.  The register is the
    running double sum of 1 / ratio (np.cumsum adds in order, as the loop does); ``exact_positions`` uses t * sr_orig /
    sr_new instead (the mistake)."""
    ratio = float(sr_new) / sr_orig
    scale = min(1.0, ratio)
    if exact_positions:
        t = np.arange(count, dtype=np.int64)
        reg = (t * sr_orig // sr_new) + (t * sr_orig % sr_new) / sr_new
    else:
        inc = np.full(count, 1.0 / ratio)
        if count:
            inc[0] = 0.0
        reg = np.cumsum(inc)
    n = reg.astype(np.int64)
    frac = scale * (reg - n)
    index_frac = frac * NUM_TABLE
    off_l = index_frac.astype(np.int64)
    eta_l = index_frac - off_l
    frac = scale - frac
    index_frac = frac * NUM_TABLE
    off_r = index_frac.astype(np.int64)
    eta_r = index_frac - off_r
    return n, off_l, eta_l, off_r, eta_r


def output_length(L, sr_orig, sr_new):
    return int(np.ceil(L * (float(sr_new) / sr_orig)))


def resample_f(x, sr_orig, sr_new, exact_positions=False, exact_step=False, with_abs=False, chunk=8192):
    """resampy's resample_f on one float64 signal: int(L * ratio) outputs.  ``with_abs`` also returns sum |w| |x| per
    output, the scale of an fp32 result's rounding error."""
    x = np.asarray(x, np.float64)
    L = x.size
    ratio = float(sr_new) / sr_orig
    n_out = int(L * ratio)
    win, delta = tables(sr_orig, sr_new)
    nwin = win.size
    step = index_step(sr_orig, sr_new, exact_step)
    taps = int(nwin // step) + 1
    n, off_l, eta_l, off_r, eta_r = positions(sr_orig, sr_new, n_out, exact_positions)
    xp = np.concatenate([np.zeros(taps + 1), x, np.zeros(taps + 1)])   # samples outside [0, L) contribute nothing
    y = np.zeros(n_out)
    s = np.zeros(n_out)
    i = np.arange(taps)
    for a in range(0, n_out, chunk):
        b = min(n_out, a + chunk)
        acc = np.zeros(b - a)
        acc_abs = np.zeros(b - a)
        for off, eta, sign in ((off_l[a:b], eta_l[a:b], -1), (off_r[a:b], eta_r[a:b], 1)):
            pos = off[:, None] + i[None, :] * step
            count = ((nwin - off) // step)[:, None]
            ok = i[None, :] < count
            idx = np.where(ok, pos, 0).astype(np.int64)
            w = np.where(ok, win[idx] + eta[:, None] * delta[idx], 0.0)
            j = n[a:b, None] + (-i[None, :] if sign < 0 else i[None, :] + 1)
            xv = xp[j + taps + 1]
            acc += (w * xv).sum(axis=1)
            acc_abs += (np.abs(w) * np.abs(xv)).sum(axis=1)
        y[a:b] = acc
        s[a:b] = acc_abs
    return (y, s) if with_abs else y


def resample(x, sr_orig, sr_new, length="ceil", **mistakes):
    """librosa.core.resample(x, sr_orig, sr_new, res_type='kaiser_best', fix=True) in float64.  ``length='int'`` returns
    resampy's int(L * ratio) samples without fix_length's zero (the mistake)."""
    x = np.asarray(x, np.float64)
    if sr_orig == sr_new:
        return x.copy()
    y = resample_f(x, sr_orig, sr_new, **mistakes)
    if length == "ceil":
        y = np.concatenate([y, np.zeros(output_length(x.size, sr_orig, sr_new) - y.size)])
    return y


def pcm_to_float(pcm, channels):
    """librosa.load's samples before resampling: audioread's float32(pcm) * (1 / 32768), channels mixed with np.mean."""
    y = np.float32(1.0 / 32768) * np.asarray(pcm, "<i2").astype(np.float32)
    if channels > 1:
        y = np.mean(y.reshape((-1, channels)).T, axis=0)
    return y


# ---- the accuracy bound of the GPU tests ---------------------------------------------------------------------------
# An fp32 output is within c * sum |w| |x| + 2^-24 |y| of float64; c = C_BOUND.  Measured on a B200 (1000 W limit) over
# every rate, signal and length of tests/test_gpu_resample.py: c = 4.48e-7 at most (noise 16 -> 20 kHz; sine 2.43e-7,
# chirp 3.92e-7, silence exact).  The bound is about 2x that.
C_BOUND = 1e-6


def error_ratio(got, want, abs_sum):
    """Largest (|got - want| - 2^-24 |want|) / sum |w| |x|: the c an fp32 result needs to stay inside the bound.  inf
    where sum |w| |x| is 0 (padding, silence) and got != want."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    excess = np.maximum(np.abs(got - want) - 2.0 ** -24 * np.abs(want), 0.0)
    ratio = np.where(abs_sum > 0, excess / np.where(abs_sum > 0, abs_sum, 1.0), np.where(excess > 0, np.inf, 0.0))
    return float(ratio.max()) if ratio.size else 0.0


def make_signal(kind, L, seed, sample_rate):
    """Seeded float32 test signals at ``sample_rate``: 'silence', 'sine' (full scale, 440 Hz), 'noise', 'chirp'
    (60 Hz up to 0.45 sample_rate)."""
    rng = np.random.default_rng(seed)
    t = np.arange(L) / sample_rate
    if kind == "silence":
        y = np.zeros(L)
    elif kind == "sine":
        y = 0.999 * np.sin(2 * np.pi * 440.0 * t + rng.uniform(0, 2 * np.pi))
    elif kind == "noise":
        y = rng.uniform(-0.5, 0.5, L)
    elif kind == "chirp":
        y = 0.8 * scipy.signal.chirp(t, f0=60.0, t1=max(L / sample_rate, 1e-3), f1=0.45 * sample_rate)
    else:
        raise ValueError(kind)
    return y.astype(np.float32)


def period(sr_orig, sr_new):
    """p of the reduced ratio p / q = sr_new / sr_orig: outputs per period of the phase pattern."""
    return sr_new // math.gcd(sr_orig, sr_new)
