"""The float64 duration search (tests/alignment_oracle.py) on the CPU: optimality against every monotonic path, known
answers, and that the two conventions most easily misread (ties, the band) each change a known answer."""
import itertools

import numpy as np
import pytest

import alignment_oracle as A


def all_paths(X, Y):
    """Every monotonic path from symbol 0 to X - 1 over Y steps, one step at most per step, each symbol at least once."""
    for moves in itertools.combinations(range(1, Y), X - 1):
        path, x = [], 0
        for y in range(Y):
            if x < X - 1 and y in moves:
                x += 1
            path.append(x)
        yield np.asarray(path)


@pytest.mark.parametrize("X,Y", [(X, Y) for X in (1, 2, 3, 4, 6) for Y in (1, 2, 5, 7, 10) if Y >= X])
@pytest.mark.parametrize("kind", ["random", "coarse"])
def test_optimum_equals_brute_force(X, Y, kind):
    rng = np.random.default_rng(100 * X + Y)
    for trial in range(5):
        if kind == "random":
            a = rng.dirichlet(np.ones(X + 2), Y + 3).T.astype(np.float32)     # columns sum to 1, padded rows / cols
        else:
            a = rng.choice(np.float32([0.0, 0.25, 0.5]), (X + 2, Y + 3))      # ties and underflowed zeros
        s = A.scores(a, X, Y)
        best = max(A.path_score(s, p) for p in all_paths(X, Y))
        d, path, Q = A.durations(a, X, Y, 1)
        assert Q[Y - 1, X - 1] == best
        assert A.path_score(s, path) == best
        assert np.array_equal(A.path_from_durations(d, X, Y, 1), path)


@pytest.mark.parametrize("r", [1, 2, 5])
def test_one_step_per_symbol_when_steps_equal_symbols(r):
    rng = np.random.default_rng(r)
    for X in (1, 2, 7, 31):
        a = rng.random((X + 1, X + 4)).astype(np.float32)
        for F in range((X - 1) * r + 1, X * r + 1):                          # Y == X for every residue
            d, path, _ = A.durations(a, X, F, r)
            assert np.array_equal(path, np.arange(X))
            assert list(d[:X]) == [r] * (X - 1) + [F - (X - 1) * r] and not d[X:].any()


@pytest.mark.parametrize("r", [1, 3, 5])
def test_uniform_matrix_stays_on_ties(r):
    for X, Y in ((1, 9), (2, 2), (3, 11), (8, 40), (33, 100)):
        for F in range((Y - 1) * r + 1, Y * r + 1):
            a = np.full((X + 3, Y + 2), 1.0 / X, np.float32)
            d, _, _ = A.durations(a, X, F, r)
            assert list(d[:X]) == [r] * (X - 1) + [F - (X - 1) * r], (X, Y, F)


def test_last_step_is_truncated():
    X, r = 3, 5
    a = np.full((X, 10), 0.5, np.float32)
    for F, want in ((21, [5, 5, 11]), (22, [5, 5, 12]), (25, [5, 5, 15]), (11, [5, 5, 1])):
        d, _, _ = A.durations(a, X, F, r)
        assert list(d) == want and sum(want) == F
    assert list(A.frames_of_steps(23, 5)) == [5, 5, 5, 5, 3]


@pytest.mark.parametrize("X,Y", [(1, 1), (1, 30), (5, 5), (5, 60), (40, 41), (64, 500)])
def test_planted_path_is_recovered(X, Y):
    rng = np.random.default_rng(X * Y)
    for r in (1, 5):
        planted = A.planted_path(rng, X, Y)
        a = np.full((X + 2, Y + 2), 1e-3, np.float32)
        a[planted, np.arange(Y)] = 0.9
        F = Y * r - rng.integers(0, r)
        d, path, _ = A.durations(a, X, F, r)
        assert np.array_equal(path, planted)
        assert np.array_equal(d, A.durations_of_path(planted, F, r, X + 2))


def test_padding_is_never_read():
    rng = np.random.default_rng(5)
    X, Y, r = 6, 20, 2
    a = rng.random((X + 4, Y + 6)).astype(np.float32)
    b = a.copy()
    b[X:], b[:, Y:] = np.nan, np.nan
    for F in (2 * Y - 1, 2 * Y):
        assert np.array_equal(A.durations(a, X, F, r)[0], A.durations(b, X, F, r)[0])


def test_zero_weights_score_as_the_smallest_float():
    assert A.scores(np.zeros((1, 1), np.float32), 1, 1)[0, 0] == np.log(2.0 ** -149)


def test_mutations_change_the_uniform_answer():
    X, Y, r = 4, 10, 5
    F = Y * r - 2
    a = np.full((X, Y), 1.0 / X, np.float32)
    want = [r] * (X - 1) + [F - (X - 1) * r]
    assert list(A.durations(a, X, F, r)[0]) == want
    assert want == [5, 5, 5, 33]
    assert list(A.durations(a, X, F, r, advance_on_tie=True)[0]) == [35, 5, 5, 3]   # the path leaves the end at once
    assert list(A.durations(a, X, F, r, band=False)[0]) == [0, 0, 0, 48]           # nothing forces a step per symbol
