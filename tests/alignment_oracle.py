"""Float64 numpy restatement of per-symbol durations from a teacher-forced alignment (``taco_durations``).

The search is Glow-TTS's ``monotonic_align.maximum_path`` (recurrence, band, tie rule; restated from memory of that code,
which is not installed here, so unpinned), accumulated in float64.  For one utterance with alignment ``a [T_in, steps]``
(``a[x, y]``: symbol x, decoder step y), ``X`` symbols and ``F`` target frames, ``Y = ceil(F / r)`` steps:

* score ``s[y][x] = log(max((double) a[x, y], 2^-149))``;
* band ``max(0, X + y - Y) <= x <= min(X - 1, y)``;
* ``Q[0][0] = s[0][0]``; ``Q[y][x] = s[y][x] + max(stay, adv)``, ``stay = Q[y-1][x]`` (-inf when x == y),
  ``adv = Q[y-1][x-1]`` (-inf when x == 0);
* backtrack from ``x = X - 1``: for y = Y - 1 .. 0, ``path[y] = x``, then ``x -= 1`` if ``x != 0`` and (``x == y`` or
  ``Q[y-1][x] < Q[y-1][x-1]``) -- a tie stays on the symbol;
* step y covers ``min(r, F - y r)`` frames; ``d[x]`` sums them over the steps on x, ``d[x] = 0`` for ``x >= X``.

``advance_on_tie`` and ``band=False`` are deliberate mistakes for the tests' mutation check."""
import numpy as np

TINY = 2.0 ** -149
NEG = -np.inf


def steps_for(F, r):
    return -(-int(F) // int(r))


def scores(a, X, Y):
    """``s [Y, X]`` float64 from the alignment rows < X and columns < Y (nothing else is read)."""
    a = np.asarray(a)[:X, :Y].astype(np.float64)
    return np.log(np.maximum(a, TINY)).T


def forward(s, band=True):
    """``Q [Y, X]`` of the recurrence; -inf outside the band.  ``band=False`` drops the band: every symbol of every
    step is computed, row 0 starts anywhere and a symbol may stay at x == y."""
    Y, X = s.shape
    Q = np.full((Y, X), NEG)
    if band:
        Q[0, 0] = s[0, 0]
    else:
        Q[0] = s[0]
    xs = np.arange(X)
    for y in range(1, Y):
        prev = Q[y - 1]
        stay = prev.copy()
        if band:
            stay[xs == y] = NEG
        adv = np.concatenate([[NEG], prev[:-1]])
        lo, hi = (max(0, X + y - Y), min(X - 1, y)) if band else (0, X - 1)
        Q[y, lo:hi + 1] = s[y, lo:hi + 1] + np.maximum(stay[lo:hi + 1], adv[lo:hi + 1])
    return Q


def backtrack(Q, advance_on_tie=False, band=True):
    """``path [Y]``: the symbol of every step."""
    Y, X = Q.shape
    path = np.zeros(Y, np.int64)
    x = X - 1
    for y in range(Y - 1, -1, -1):
        path[y] = x
        if x != 0 and y > 0:
            a, b = Q[y - 1, x], Q[y - 1, x - 1]
            if (band and x == y) or (a <= b if advance_on_tie else a < b):
                x -= 1
    return path


def frames_of_steps(F, r):
    Y = steps_for(F, r)
    return np.minimum(r, F - np.arange(Y) * r)


def durations_of_path(path, F, r, T_in):
    d = np.zeros(T_in, np.int64)
    np.add.at(d, path, frames_of_steps(F, r))
    return d.astype(np.int32)


def durations(a, X, F, r, advance_on_tie=False, band=True):
    """``(d int32 [T_in], path [Y], Q [Y, X])`` of one utterance ``a [T_in, steps]``."""
    Y = steps_for(F, r)
    Q = forward(scores(a, X, Y), band=band)
    path = backtrack(Q, advance_on_tie=advance_on_tie, band=band)
    return durations_of_path(path, F, r, np.asarray(a).shape[0]), path, Q


def path_from_durations(d, X, F, r):
    """The step path that durations ``d`` describe; raises AssertionError unless ``d`` is a monotonic path in the band:
    every symbol < X at least one step, whole steps of r frames except the last step's ``F - (Y - 1) r``, sum F, zeros
    past X."""
    d = np.asarray(d, np.int64)
    Y = steps_for(F, r)
    assert d.sum() == F and (d[:X] >= 1).all() and not d[X:].any(), (d, X, F)
    last = F - (Y - 1) * r
    assert (d[:X - 1] % r == 0).all() and (d[X - 1] - last) % r == 0 and d[X - 1] >= last, (d, X, F, r)
    n = d[:X] // r
    n[X - 1] = (d[X - 1] - last) // r + 1
    return np.repeat(np.arange(X), n)


def path_score(s, path):
    """Sum of ``s[y, path[y]]`` in step order (float64), the order in which Q accumulates."""
    total = 0.0
    for y, x in enumerate(path):
        total = float(s[y, x]) + total
    return total


def planted_path(rng, X, Y):
    """A random monotonic path from symbol 0 to X - 1 over Y steps, every symbol at least one step."""
    cuts = np.sort(rng.choice(np.arange(1, Y), X - 1, replace=False)) if X > 1 else np.zeros(0, np.int64)
    return np.repeat(np.arange(X), np.diff(np.concatenate([[0], cuts, [Y]])))
