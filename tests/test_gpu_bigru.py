"""The two BiGRU recurrence kernels called directly (``taco_bigru_unit``): ``bigru_kernel<NS>`` (impl 0, fp32 FFMA, the
default; NS = 1 / 2 / 4 utterances per CTA for N <= 74 / <= 148 / more) and ``bigru_mma_kernel`` (impl 1, mma.sync on
bf16 hi/lo operands, 8 utterances per CTA), against the float64 step of ``tests/bigru_oracle.py``.

Accuracy is checked step by step (``local_check``): every output element of every valid step against one float64 GRU
step from the kernel's own previous state, with the first-order per-element bound of the oracle module.  Constants:

* ``C_FFMA`` (impl 0): relative error of the fp32 dot products.  Its errors are at the fp32 rounding of the output: with
  eps_act = 2e-7 the worst element needs c = 1.8e-6, with 5e-7 it needs 3.4e-9.  C_FFMA = 3e-6.
* ``C_MMA`` (impl 1): relative error of the bf16x3 dot products (hh + hl + lh).  Worst needed c with eps_act = 5e-7: 1.96e-6
  (2.1e-6 with 2e-7).  C_MMA = 6e-6.  A kernel without the hl product needs 3.5e-4 ... 7.5e-4 and fails.
* ``EPS_ACT`` = 5e-7: absolute error of ``ex2.approx`` / ``rcp.approx`` in sigmoid / tanh and of the state update.  Both
  kernels stay within 2e-7 at the c above.

Measured on an NVIDIA B200 (1000 W power limit) over the geometries and inputs below.

Inputs: the recurrent kernels of both CBHGs at random init (contracting) and scaled by 4 (not contracting, gates
saturating), xproj ~ N(0, 1) and the same with a tenth of its entries at +-30; lengths 0, 1, 2, T-1 and T mixed inside every
CTA.  Every call writes into a NaN-filled buffer one utterance wider on each side than its output.

Exact checks: with update pre-activations at -1000 / +1000 the kernels compute u = 0 / 1 exactly, and with candidate
pre-activations at +-1000 tanh = +-1 exactly (2^+-big saturates, rcp(inf) = 0), so the output is a known sign pattern bit for
bit; a batch equals its utterances run alone (impl 0) or in any CTA column (impl 1); repeated calls give the same bits.
"""
import numpy as np
import pytest
import torch

import bigru_oracle as B

pytestmark = pytest.mark.gpu

C_FFMA = 3e-6      # measured 1.8e-6 at eps_act 2e-7 (module docstring)
C_MMA = 6e-6       # measured 1.96e-6 at eps_act 5e-7
EPS_ACT = 5e-7     # measured <= 2e-7 for both kernels
C_X3 = 2.5e-5       # the tcgen05 GEMM in bf16x3 mode (tests/test_gpu_umma.py)
C_ROUND = 1e-6      # its fp32 epilogue (bias add, store)
NAN32 = 0x7FC0DEAD  # quiet NaN with a payload no kernel writes
SAT = 1000.0        # pre-activation that saturates sigmoid / tanh exactly whatever h U adds (|h| <= 1)
SCOPES = ["encoder_cbhg", "post_cbhg"]
C_OF = {0: C_FFMA, 1: C_MMA}

FFMA_N = [1, 2, 74, 75, 148, 149, 256]
MMA_N = [1, 7, 8, 9, 16, 33]
TS = [1, 2, 31, 1000]
GEOMS = ([(0, n, t) for n in FFMA_N for t in TS] + [(0, 2, 2000)] +
         [(1, n, t) for n in MMA_N for t in TS] + [(1, 9, 2000)])
VARIANTS = [(s, k, x) for s in SCOPES for k in (1.0, 4.0) for x in ("normal", "spiky")]


@pytest.fixture(scope="module")
def eng(small_hp, small_weights):
    from tacotron_multispeaker_b200.engine import Engine
    e = Engine(small_hp, id_num=6)
    e.load_weights(small_weights)
    yield e
    e.close()


@pytest.fixture(scope="module")
def rec(small_weights):
    """scope -> (wx, bx, ug, uc) as the kernels read them."""
    return {s: B.split_weights(small_weights, s) for s in SCOPES}


@pytest.fixture(scope="module")
def stats():
    """Worst c / eps_act each kernel needed over the module's accuracy tests (printed at the end: ``pytest -s``)."""
    st = {0: [0.0, 0.0, {}], 1: [0.0, 0.0, {}]}
    yield st
    for impl, (c, e, grid) in st.items():
        print("\nbigru impl %d: worst needed c %.3e (C = %.1e, ratio %.3f), eps_act %.3e (EPS_ACT = %.1e, ratio %.3f); c at eps %s"
              % (impl, c, C_OF[impl], c / C_OF[impl], e, EPS_ACT, e / EPS_ACT, grid))


def lengths_for(N, T, seed=0):
    """0, 1, 2, T-1, T in turn (clipped to T), so every CTA of 2, 4 or 8 utterances mixes them; every 7th a random one."""
    base = np.array([T, 0, 1, 2, T - 1])
    L = np.minimum(base[np.arange(N) % 5], T)
    rng = np.random.default_rng(seed + N * 7 + T)
    if T > 4:
        L[6::7] = rng.integers(3, T - 1, len(L[6::7]))
    return L.astype(np.int32)


def make_xproj(N, T, kind, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((N, T, 768)).astype(np.float32)
    if kind == "spiky":
        m = rng.random((N, T, 768)) < 0.1
        x[m] = np.where(rng.random(int(m.sum())) < 0.5, -30.0, 30.0)
    return x


def guarded(N, T):
    """(buffer [N+2, T, 256] of NaN bits, the output view buffer[1:N+1])."""
    buf = torch.full((N + 2, T, 256), 0, dtype=torch.int32, device="cuda")
    buf.fill_(NAN32)
    return buf, buf.view(torch.float32)[1:N + 1]


def check_window(buf, out, lengths):
    """Every element of the output written (finite), exactly zero past each length; the guard utterances keep their NaN bits."""
    g = buf.cpu()
    assert bool((g[0] == NAN32).all()) and bool((g[-1] == NAN32).all()), "a write outside the output"
    o = out.cpu()
    assert bool(torch.isfinite(o).all()), "an output element not written"
    for n, L in enumerate(lengths):
        assert bool((o[n, int(L):] == 0).all()), "nonzero output past length %d of utterance %d" % (L, n)


def run(eng, impl, xproj_np, lengths, ug, uc):
    N, T, _ = xproj_np.shape
    buf, out = guarded(N, T)
    xp = torch.from_numpy(xproj_np).cuda()
    eng.bigru_unit(xp, ug, uc, lengths, impl=impl, out=out)
    torch.cuda.synchronize()
    return buf, out


# ---------------------------------------------------------------------------------------------------------------------
# local accuracy at every geometry, lengths and weight regime
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl,N,T", GEOMS, ids=["impl%d-N%d-T%d" % g for g in GEOMS])
def test_local_accuracy(eng, rec, stats, impl, N, T):
    lengths = lengths_for(N, T)
    gi = GEOMS.index((impl, N, T))
    variants = VARIANTS if T <= 31 else [VARIANTS[(2 * gi) % 8], VARIANTS[(2 * gi + 5) % 8]]
    for vi, (scope, k, kind) in enumerate(variants):
        _, _, ug, uc = rec[scope]
        ug, uc = ug * np.float32(k), uc * np.float32(k)
        xproj = make_xproj(N, T, kind, seed=gi * 10 + vi)
        buf, out = run(eng, impl, xproj, lengths, ug, uc)
        check_window(buf, out, lengths)
        r = B.local_check(out.cpu().numpy(), xproj, lengths, ug, uc, C_OF[impl], EPS_ACT)
        st = stats[impl]
        st[0], st[1] = max(st[0], r.c_ratio), max(st[1], r.eps_excess)
        for e, v in r.c_at_eps.items():
            st[2][e] = max(st[2].get(e, 0.0), v)
        print("impl %d N %d T %d %s x%g %s: %s" % (impl, N, T, scope, k, kind, r))
        assert r.ok, "impl %d N %d T %d %s x%g %s: %s" % (impl, N, T, scope, k, kind, r)


# ---------------------------------------------------------------------------------------------------------------------
# exact mapping: saturated gates give a known sign pattern bit for bit
# ---------------------------------------------------------------------------------------------------------------------
def kat_case(N, T, lengths, seed):
    """xproj with u = 0 (write: state := +-1) or u = 1 (carry: state kept) per element, and the outputs that implies."""
    rng = np.random.default_rng(seed)
    carry = rng.random((N, T, 2, 128)) < 0.3
    sgn = np.where(rng.random((N, T, 2, 128)) < 0.5, -1.0, 1.0).astype(np.float32)
    xproj = np.zeros((N, T, 768), np.float32)
    for d in range(2):
        o = d * 384
        xproj[..., o:o + 128] = rng.standard_normal((N, T, 128))          # reset gate: irrelevant once tanh saturates
        xproj[..., o + 128:o + 256] = np.where(carry[:, :, d], SAT, -SAT)
        xproj[..., o + 256:o + 384] = SAT * sgn[:, :, d]
    want = np.zeros((N, T, 256), np.float32)
    ar = np.arange(N)
    for d in range(2):
        h = np.zeros((N, 128), np.float32)
        for s in range(int(lengths.max(initial=0))):
            live = s < lengths
            p = np.clip(s if d == 0 else lengths - 1 - s, 0, T - 1) * np.ones(N, np.int64)
            hn = np.where(carry[ar, p, d], h, sgn[ar, p, d])
            h = np.where(live[:, None], hn, h)
            cur = want[ar, p, d * 128:(d + 1) * 128]
            want[ar, p, d * 128:(d + 1) * 128] = np.where(live[:, None], hn, cur)
    return xproj, want


@pytest.mark.parametrize("impl,N,T", GEOMS, ids=["impl%d-N%d-T%d" % g for g in GEOMS])
def test_saturated_gates_exact_mapping(eng, rec, impl, N, T):
    """Catches a misplaced utterance, column, position, direction or ring slot exactly: out[n, p, 128 dir + j] is the sign
    written at the last step of that direction that had u = 0 in column j (0 before any), bit for bit."""
    _, _, ug, uc = rec["post_cbhg" if N % 2 else "encoder_cbhg"]
    assert np.abs(ug).sum(axis=1).max() < SAT / 10 and np.abs(uc).sum(axis=1).max() < SAT / 10
    lengths = lengths_for(N, T, seed=1)
    xproj, want = kat_case(N, T, lengths, seed=N * 13 + T)
    buf, out = run(eng, impl, xproj, lengths, ug, uc)
    check_window(buf, out, lengths)
    got = out.cpu().numpy()
    bad = np.argwhere(got != want)
    assert bad.size == 0, "first mismatch (n, p, col) %s: got %r want %r (%d elements)" % (
        tuple(bad[0]), got[tuple(bad[0])], want[tuple(bad[0])], len(bad))


# ---------------------------------------------------------------------------------------------------------------------
# independence and repeatability
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,T", [(75, 40), (149, 40), (256, 31)])
def test_ffma_batch_equals_single_utterances(eng, rec, N, T):
    """impl 0: the per-utterance arithmetic does not depend on NS or on the slot in the CTA, so a batch (NS = 2 / 4) equals
    its utterances run one by one (NS = 1) bit for bit."""
    _, _, ug, uc = rec["post_cbhg"]
    ug, uc = ug * np.float32(4.0), uc * np.float32(4.0)
    lengths = lengths_for(N, T, seed=2)
    xproj = make_xproj(N, T, "spiky", seed=N)
    _, out = run(eng, 0, xproj, lengths, ug, uc)
    xp = torch.from_numpy(xproj).cuda()
    single = torch.empty_like(out)
    for n in range(N):
        eng.bigru_unit(xp[n:n + 1], ug, uc, lengths[n:n + 1], impl=0, out=single[n:n + 1])
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int32), single.view(torch.int32))


@pytest.mark.parametrize("T", [31, 300])
def test_mma_column_does_not_matter(eng, rec, T):
    """impl 1: an utterance gives the same bits in any of the 8 columns of a CTA, and in the second CTA of a batch."""
    _, _, ug, uc = rec["encoder_cbhg"]
    lengths = lengths_for(8, T, seed=3)
    xproj = make_xproj(8, T, "normal", seed=T)
    _, base = run(eng, 1, xproj, lengths, ug, uc)
    base = base.cpu()
    for rot in range(1, 8):
        perm = (np.arange(8) + rot) % 8
        xp2 = np.concatenate([xproj[perm[::-1]], xproj[perm]])         # 16 utterances: two CTAs, two column orders
        _, got = run(eng, 1, np.ascontiguousarray(xp2), np.concatenate([lengths[perm[::-1]], lengths[perm]]), ug, uc)
        got = got.cpu()
        rev = torch.from_numpy(perm[::-1].copy())
        assert torch.equal(got[:8].view(torch.int32), base[rev].view(torch.int32)), rot
        assert torch.equal(got[8:].view(torch.int32), base[torch.from_numpy(perm)].view(torch.int32)), rot


@pytest.mark.parametrize("impl,N,T", [(0, 149, 200), (1, 33, 200)])
def test_repeated_calls_bit_identical(eng, rec, impl, N, T):
    _, _, ug, uc = rec["post_cbhg"]
    lengths = lengths_for(N, T, seed=4)
    xproj = make_xproj(N, T, "spiky", seed=5)
    outs = [run(eng, impl, xproj, lengths, ug, uc)[1].cpu() for _ in range(3)]
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))
    assert torch.equal(outs[0].view(torch.int32), outs[2].view(torch.int32))


# ---------------------------------------------------------------------------------------------------------------------
# the production entry at the config-4 shape
# ---------------------------------------------------------------------------------------------------------------------
def test_production_entry_post_cbhg_n256_t1000(eng, rec, monkeypatch):
    """``Engine.bigru`` (tensor-core GEMM for xproj, then the default FFMA recurrence) on the post-net CBHG at N = 256,
    T = 1000, checked against the float64 xproj with the GEMM's error bound C_X3 sum |x||Wx| + C_ROUND |xproj| added to the
    pre-activation errors."""
    monkeypatch.delenv("TACO_BIGRU", raising=False)
    N, T = 256, 1000
    wx, bx, ug, uc = rec["post_cbhg"]
    lengths = lengths_for(N, T, seed=6)
    rng = np.random.default_rng(7)
    x = rng.standard_normal((N, T, 128)).astype(np.float32)
    out = eng.bigru(1, x, lengths).cpu().numpy()
    xt = torch.from_numpy(x).cuda().double()
    xproj = (xt @ torch.from_numpy(wx).cuda().double() + torch.from_numpy(bx).cuda().double())
    xerr = C_X3 * (xt.abs() @ torch.from_numpy(wx).cuda().double().abs()) + C_ROUND * xproj.abs()
    xproj, xerr = xproj.cpu().numpy(), xerr.float().cpu().numpy()
    r = B.local_check(out, xproj, lengths, ug, uc, C_FFMA, EPS_ACT, xproj_err=xerr)
    print("production N %d T %d: %s" % (N, T, r))
    assert r.ok, str(r)
    for n, L in enumerate(lengths):
        assert np.all(out[n, L:] == 0.0)


# ---------------------------------------------------------------------------------------------------------------------
# refusals
# ---------------------------------------------------------------------------------------------------------------------
def test_refusals(eng, rec):
    from tacotron_multispeaker_b200._abi import TACO_ERR_INVALID
    lib = eng.lib
    _, _, ug, uc = rec["encoder_cbhg"]
    xp = torch.zeros(2, 4, 768 + 4, device="cuda")
    out = torch.zeros(2, 4, 256 + 4, device="cuda")
    X, O = xp.data_ptr(), out.data_ptr()
    g, c = ug.ctypes.data, uc.ctypes.data
    st = eng.stream

    def call(impl=0, x=X, N=2, T=4, ugp=g, ucp=c, o=O, h=None):
        return lib.taco_bigru_unit(eng._h if h is None else h, impl, x, None, N, T, ugp, ucp, o, st)

    assert call() == 0 and call(impl=1) == 0
    torch.cuda.synchronize()
    for kw in (dict(impl=2), dict(impl=-1), dict(N=0), dict(N=-1), dict(T=0), dict(T=-5), dict(x=None), dict(ugp=None),
               dict(ucp=None), dict(o=None), dict(x=X + 4), dict(o=O + 8)):
        assert call(**kw) == TACO_ERR_INVALID, kw
    assert lib.taco_bigru_unit(None, 0, X, None, 2, 4, g, c, O, st) == TACO_ERR_INVALID
