"""The float64 BiGRU restatement of ``tests/bigru_oracle.py`` against the CPU oracle, and its step-local check.  No GPU."""
import numpy as np
import pytest
import torch

import bigru_oracle as B
from oracle import taco_oracle as O

SCOPES = ["encoder_cbhg", "post_cbhg"]


def _batch(N, T, masked, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((N, T, 128)).astype(np.float32)
    lengths = None
    if masked:
        lengths = rng.integers(1, T + 1, N).astype(np.int32)
        lengths[0] = T
        lengths[-1] = 1
    return x, lengths


@pytest.mark.parametrize("scope", SCOPES)
@pytest.mark.parametrize("N,T,masked", [(1, 7, False), (3, 12, True), (5, 9, True), (2, 16, False)])
def test_bigru64_equals_oracle_in_float64(small_weights, scope, N, T, masked):
    """bigru64 on xproj = x Wx + b equals the oracle's GRUCell-by-GRUCell bigru run in float64: ties the restatement (and the
    kernels' split of the TF kernels into hoisted and recurrent halves) to the oracle the KATs pin."""
    x, lengths = _batch(N, T, masked, N * 31 + T)
    wx, bx, ug, uc = B.split_weights(small_weights, scope)
    xproj = x.astype(np.float64) @ wx.astype(np.float64) + bx.astype(np.float64)
    got = B.bigru64(xproj, lengths, ug, uc)
    ref = O.bigru(torch.from_numpy(x).double(), lengths, O.W(small_weights, torch.float64), scope).numpy()
    assert np.abs(got - ref).max() < 1e-12
    if masked:
        for n in range(N):
            assert np.all(got[n, lengths[n]:] == 0.0)


def test_gru_step64_reset_before_candidate_matmul():
    """GRUCell applies r to the state before the candidate matmul: with Uc = I, xc = 0, xg = 0 (r = u = 1/2) and h = 1,
    cand = tanh(1/2), not tanh(1) / 2."""
    h = np.ones((2, 128))
    xg, xc = np.zeros((2, 256)), np.zeros((2, 128))
    got = B.gru_step64(h, xg, xc, np.zeros((128, 256)), np.eye(128))
    assert np.allclose(got, 0.5 + 0.5 * np.tanh(0.5), rtol=0, atol=1e-15)


def _case(seed, N=6, T=11):
    rng = np.random.default_rng(seed)
    xproj = rng.standard_normal((N, T, 768))
    ug = rng.uniform(-0.2, 0.2, (2, 128, 256))
    uc = rng.uniform(-0.2, 0.2, (2, 128, 128))
    lengths = np.array([T, 0, 1, 2, T - 1, 5][:N], np.int32)
    return xproj, lengths, ug, uc


def test_local_check_accepts_own_trajectory_with_zero_bound():
    xproj, lengths, ug, uc = _case(1)
    out = B.bigru64(xproj, lengths, ug, uc)
    r = B.local_check(out, xproj, lengths, ug, uc, c=0.0, eps_act=0.0, chunk=4)
    assert r.ok, str(r)
    assert r.max_err == 0.0
    assert r.checked == 2 * 128 * int(np.sum(lengths))


@pytest.mark.parametrize("where", ["fw_first", "fw_mid", "bw_first", "bw_last", "utt1_len1"])
def test_local_check_rejects_one_perturbed_element(where):
    """One element off by 1e-9 fails the zero bound and the realistic one at 1e-3; the worst element is the one changed
    (or the step that read it as its state)."""
    xproj, lengths, ug, uc = _case(2)
    out = B.bigru64(xproj, lengths, ug, uc)
    n, p, col = {"fw_first": (0, 0, 3), "fw_mid": (0, 5, 127), "bw_first": (4, 9, 128 + 7), "bw_last": (0, 0, 255),
                 "utt1_len1": (2, 0, 200)}[where]
    assert p < lengths[n]
    for delta, c, eps in ((1e-9, 0.0, 0.0), (1e-3, 1e-6, 1e-6)):
        bad = out.copy()
        bad[n, p, col] += delta
        r = B.local_check(bad, xproj, lengths, ug, uc, c=c, eps_act=eps, chunk=4)
        assert not r.ok
        assert r.worst[0] == n and r.worst[2] == col // 128
    assert B.local_check(out, xproj, lengths, ug, uc, c=1e-6, eps_act=1e-6).ok


def test_local_check_rejects_nan():
    xproj, lengths, ug, uc = _case(3)
    out = B.bigru64(xproj, lengths, ug, uc)
    out[5, 4, 17] = np.nan
    r = B.local_check(out, xproj, lengths, ug, uc, c=1.0, eps_act=1.0)
    assert not r.ok and r.max_err == np.inf


def test_local_check_bound_is_first_order_in_the_dot_product_error():
    """A trajectory whose every pre-activation carries a relative error e passes at c = 2e and fails at c = e / 10:
    the bound is neither vacuous nor tighter than the arithmetic it describes."""
    xproj, lengths, ug, uc = _case(4)
    e = 1e-5
    rng = np.random.default_rng(5)
    out = np.zeros((6, 11, 256))
    for d in range(2):   # run the recurrence with perturbed dot products, column by column
        for n in range(6):
            h = np.zeros((1, 128))
            L = lengths[n]
            for s in range(L):
                p = s if d == 0 else L - 1 - s
                x = xproj[n, p, d * 384:(d + 1) * 384]
                hu = h @ ug[d]
                pg = x[:256] + hu + e * (np.abs(x[:256]) + np.abs(h) @ np.abs(ug[d])) * rng.choice([-1, 1], 256)
                g = B.sigmoid(pg)
                r, u = g[:, :128], g[:, 128:]
                pc = x[256:] + (r * h) @ uc[d] + e * (np.abs(x[256:]) + (r * np.abs(h)) @ np.abs(uc[d])) * rng.choice([-1, 1], 128)
                h = u * h + (1 - u) * np.tanh(pc)
                out[n, p, d * 128:(d + 1) * 128] = h
    assert B.local_check(out, xproj, lengths, ug, uc, c=2 * e, eps_act=0.0).ok
    assert not B.local_check(out, xproj, lengths, ug, uc, c=e / 10, eps_act=0.0).ok
