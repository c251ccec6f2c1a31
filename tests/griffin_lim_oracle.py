"""Float64 restatement of one Griffin-Lim iteration (reference util/audio.py:78-91, the TF conventions of
``oracle/audio_oracle.py``) and a step-local bound for the CUDA vocoder (``gl_iter_kernel`` / ``gl_ola_kernel`` /
``gl_deemph_kernel`` in griffin_lim.cu).

TEST INFRASTRUCTURE ONLY (numpy, scipy).  One iteration depends on the current signal y_k alone:

    F_t = y_k[t hop : t hop + win] w          (periodic Hann)
    X_t = rfft(F_t, 2048)
    Y_t = S_t X_t / max(1e-8, |X_t|)
    r_t = irfft(Y_t, 2048)[:win] w
    y_{k+1} = overlap_and_add(r_t, hop)

The kernel never materialises y_k: it rebuilds each frame from the previous iteration's rows, adding the covering rows in
ascending frame order, as ``gl_ola_kernel`` does.  So the waveform ``taco_griffin_lim`` returns after k iterations (without
inverse pre-emphasis) is bit for bit the signal iteration k + 1 frames, and ``gl_local_check`` runs one float64 iteration from
the kernel's own y_k and compares it with the kernel's y_{k+1} without accumulating error over iterations.

The bound is first order in ``c``, the relative error of the kernel's float32 arithmetic per bin: the 2048-point transforms
(relative to the 1-norm of their input), the magnitudes' exp2f in ``gl_mags_kernel`` and the rsqrt of the phase step:

    e_t      = c sum_i |F_t[i]|                                      error of every bin of X_t
    delta_tb = min(2, 2 e_t / max(1e-8, |X_t[b]|))                   phase error (a unit vector moves at most 2)
    |dY_tb| <= S_tb (delta_tb + c)
    |dr_t[i]| <= w[i] / 2048 sum_b m_b (|dY_tb| + c S_tb)            m_b = 1 at DC and Nyquist, 2 elsewhere
    |dy[m]|  <= sum_{t covers m} |dr_t[m - t hop]| + 2^-22 sum_{t covers m} |r_t[m - t hop]|

The last term is the float32 synthesis window, the product that writes each row and the additions of the overlap-add.  With
delta = 0 the same bound covers the zero-phase start (iteration 0).  Bins whose |X| is within a few e_t of zero have phases
float32 cannot resolve: there delta caps at 2 and the bound is the bin's whole magnitude; ``StepCheck.capped`` reports how
often that happens, since a check in which most bins cap has no teeth.
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
from scipy.signal import lfilter

from oracle import audio_oracle as A

U = 2.0 ** -24
N_FFT = 2048


def geometry(hp):
    n_fft, hop, win = A.stft_parameters(hp)
    assert n_fft == N_FFT, n_fft
    return win, hop


def mags64(lin, hp):
    """util/audio.py:42-43: (10^(0.05 (clip(x, 0, 1) (-min_db) + min_db + ref_db)))^power, [.., T, 1025] in float64."""
    x = np.asarray(lin, np.float64)
    return np.power(A.db_to_amp(A.denormalize(x, hp) + hp.ref_level_db), hp.power)


def _ola(rows, hop):
    T, win = rows.shape
    idx = (np.arange(T)[:, None] * hop + np.arange(win)[None, :]).ravel()
    return np.bincount(idx, weights=rows.ravel(), minlength=(T - 1) * hop + win)


def _frames(y, T, win, hop):
    idx = np.arange(T)[:, None] * hop + np.arange(win)[None, :]
    return np.asarray(y, np.float64)[idx]


@dataclass
class Step:
    """One float64 iteration and what the bound needs: per frame t the windowed frame F (None for the zero-phase start), its
    transform X, the magnitudes S, the rows r and the signal y they overlap-add to."""
    F: np.ndarray | None
    X: np.ndarray | None
    S: np.ndarray
    r: np.ndarray
    y: np.ndarray
    hop: int


def _rows(Y, win):
    return np.fft.irfft(Y, N_FFT, axis=-1)[:, :win] * A.hann_periodic(win)[None, :]


def gl_start64(S, hp):
    """The zero-phase start (iteration 0): istft(S) for magnitudes S [T, 1025]."""
    win, hop = geometry(hp)
    S = np.asarray(S, np.float64)
    r = _rows(S.astype(np.complex128), win)
    return Step(None, None, S, r, _ola(r, hop), hop)


def gl_step64(y, S, hp):
    """One Griffin-Lim iteration from the signal y [(T-1) hop + win] with magnitudes S [T, 1025]."""
    win, hop = geometry(hp)
    S = np.asarray(S, np.float64)
    T = S.shape[0]
    assert len(y) == (T - 1) * hop + win, (len(y), T, hop, win)
    F = _frames(y, T, win, hop) * A.hann_periodic(win)[None, :]
    X = np.fft.rfft(F, N_FFT, axis=-1)
    r = _rows(S * (X / np.maximum(1e-8, np.abs(X))), win)
    return Step(F, X, S, r, _ola(r, hop), hop)


class _Bound:
    """gl_local_bound's pieces that do not depend on c, so that a search over c is cheap."""

    def __init__(self, st: Step):
        self.hop = st.hop
        mb = np.full(st.S.shape[-1], 2.0)
        mb[0] = mb[-1] = 1.0
        self.mS = mb * st.S                                               # m_b S_tb
        self.mS_sum = np.sum(self.mS, axis=1)
        if st.X is None:
            self.sumF = self.absX = None
        else:
            self.sumF = np.sum(np.abs(st.F), axis=1)
            self.absX = np.maximum(1e-8, np.abs(st.X))
        self.w = A.hann_periodic(st.r.shape[1])
        self.rounding = 4.0 * U * _ola(np.abs(st.r), st.hop)

    def delta(self, c):
        if self.absX is None:
            return None
        return np.minimum(2.0, (2.0 * c) * self.sumF[:, None] / self.absX)

    def __call__(self, c):
        rho = 2.0 * c * self.mS_sum
        d = self.delta(c)
        if d is not None:
            rho = rho + np.sum(self.mS * d, axis=1)
        return _ola(self.w[None, :] * (rho / N_FFT)[:, None], self.hop) + self.rounding


def gl_local_bound(st: Step, c):
    """Per-sample bound of |kernel y_{k+1} - st.y| at FFT error c (module docstring)."""
    return _Bound(st)(c)


@dataclass
class StepCheck:
    max_ratio: float       # max |got - want| / bound (inf for a NaN, or an error where the bound is 0)
    median_ratio: float    # over the samples some frame covers
    capped: float          # fraction of (frame, bin) pairs whose phase bound hit its cap of 2
    needed_c: float        # the smallest c at which every sample is within its bound (inf: none up to 1e-2)
    worst: tuple           # (sample, got, want, bound) of the largest ratio

    def __str__(self):
        return "max ratio %.3g, median %.3g, capped %.4f, needs c >= %.3g, worst (m, got, want, bound) = %s" % (
            self.max_ratio, self.median_ratio, self.capped, self.needed_c, self.worst)


def _ratio(err, bound):
    with np.errstate(divide="ignore", invalid="ignore"):
        q = np.where(bound > 0, err / bound, np.where(err > 0, np.inf, 0.0))
    return np.where(np.isnan(err), np.inf, q)


def gl_local_check(y_k, y_k1, S, hp, c, search=True):
    """Step-local check of a kernel's y_{k+1} (1-D) against one float64 iteration from its own y_k (None: y_k1 is the
    zero-phase start).  search: also find the smallest c this output needs (bisection on log c)."""
    st = gl_start64(S, hp) if y_k is None else gl_step64(np.asarray(y_k, np.float64), S, hp)
    got = np.asarray(y_k1, np.float64)
    assert got.shape == st.y.shape, (got.shape, st.y.shape)
    err = np.abs(got - st.y)
    err = np.where(np.isnan(err), np.inf, err)
    B = _Bound(st)
    bound = B(c)
    q = _ratio(err, bound)
    covered = _ola(np.ones_like(st.r), st.hop) > 0
    i = int(np.argmax(q))
    d = B.delta(c)
    capped = 0.0 if d is None else float(np.mean(d >= 2.0))
    needed = np.nan
    if search:
        if np.all(err <= B(0.0)):
            needed = 0.0
        elif not np.all(err <= B(1e-2)):
            needed = np.inf
        else:
            lo, hi = np.log(1e-12), np.log(1e-2)
            for _ in range(14):
                mid = 0.5 * (lo + hi)
                lo, hi = (lo, mid) if np.all(err <= B(np.exp(mid))) else (mid, hi)
            needed = float(np.exp(hi))
    return StepCheck(float(q[i]), float(np.median(q[covered])), capped, needed,
                     (i, float(got[i]), float(st.y[i]), float(bound[i])))


def deemph_bound(x, a, c):
    """Per-sample bound of gl_deemph_kernel's output against lfilter([1], [1, -a], x) of its own input x:
    c lfilter([1], [1, -|a|], |x|) (the scan's powers of a, products and carries) + 2^-24 |z| (the final rounding)."""
    x = np.asarray(x, np.float64)
    z = lfilter([1.0], [1.0, -a], x)
    return c * lfilter([1.0], [1.0, -abs(a)], np.abs(x)) + U * np.abs(z)


def deemph_check(got, x, a, c):
    """(max |got - inv_preemphasis(x)| / deemph_bound (inf for a NaN), the index where it is reached, the smallest c at
    which every sample is within its bound)."""
    want = A.inv_preemphasis(np.asarray(x, np.float64), _Coef(a))
    err = np.abs(np.asarray(got, np.float64) - want)
    err = np.where(np.isnan(err), np.inf, err)
    q = _ratio(err, deemph_bound(x, a, c))
    i = int(np.argmax(q))
    need = _ratio(np.maximum(0.0, err - U * np.abs(want)), deemph_bound(x, a, 1.0) - U * np.abs(want))
    return float(q[i]), i, float(np.max(need))


@dataclass
class _Coef:
    preemphasis: float
