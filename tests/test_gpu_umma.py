"""The tensor-core GEMM (``conv_umma_kernel``) and the fused highway kernel (``highway4_kernel``) called directly, against a
float64 reference of the same operation, on every launch shape and epilogue the forward uses.

Reference: ``oracle.conv1d_same`` / the highway formula on float64 copies of the fp32 inputs, then activation, affine,
residual and gate in float64.  Tolerance, per element:

    tol = c * S * max(1, |scale|) + C_ROUND * (|ref| + |res|),     S = sum_i |x_i| |w_i|   (the same conv on |x|, |w|)

so a wrong product (a dropped hi*lo term, a tap read from the wrong row) fails even where the output is small.  ``c`` depends
on the arithmetic:

* ``C_X3`` for the default bf16x3 mode (hi*hi + hi*lo + lo*hi).  Worst ratio (|got - ref| - C_ROUND (|ref| + |res|)) / (S
  max(1, |scale|)) measured on a B200 over the case table: 8.2e-6 (t1000_k8_cin4_cout768: 32-term sums, where the split error
  of single terms, up to ~3 x 2^-18, is not averaged away; 1e-6 .. 4e-6 elsewhere).  ``C_X3`` = 2.5e-5, three times that.
  A mode-2 run (one product per k-step) of every case must FAIL this bound (asserted): its smallest ratio on the table is
  2.2e-4, and a kernel without the hi*lo product measured 5.5e-4.
* ``C_BF16`` for plain bf16 (mode 2): 2^-7, the worst case of one bf16 product per term (2 x 2^-9) with margin.

Outputs are written into NaN-filled buffers wider than the written window (column offset, row pitch, batch stride and one
extra utterance): everything outside the window must still hold the NaN pattern bit for bit.

The launch plan of every case (``taco_umma_plan``) is pinned in the table; the CPU tests check the table covers every
branch of the plan, and each GPU case checks that the launch used the planned shape.
"""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

from oracle import taco_oracle as O

C_X3 = 2.5e-5      # mode 1; measured worst ratio on the case table: 8.2e-6 (module docstring)
C_BF16 = 2.0 ** -7  # mode 2
C_ROUND = 1e-6     # fp32 rounding of the epilogue (bias, activation, affine, residual, gate)
SMS = 148          # B200
NAN32 = 0x7FC0DEAD  # quiet NaN with a payload no kernel writes
NAN16 = 0x7FC1     # bf16 quiet NaN with a payload
FAKE = 0x10000     # a 16-byte aligned stand-in address for the host-only plan function

ONE, SHORT, LONG = "one tile per CTA", "persistent short K", "persistent long K"


class Case:
    def __init__(self, name, N, T, Cin, Cout, taps=1, bank=1, act=0, affine=False, res=False, layout="vec", plan=None):
        self.name, self.N, self.T, self.Cin, self.Cout, self.taps, self.bank = name, N, T, Cin, Cout, taps, bank
        self.act, self.affine, self.res, self.layout = act, affine, res, layout
        self.plan = plan          # (kind, acc_cols, vec_epi, variant)

    @property
    def width(self):              # output channels written per row
        return self.Cout * self.bank

    def geometry(self):
        """Strides of x, res and out: wider than the data, 16-byte multiples in the vector layout, odd in the scalar one."""
        v = self.layout == "vec"
        g = {}
        g["ldx"] = self.Cin + 4
        g["x_bs"] = self.T * g["ldx"] + 4
        g["ldres"] = self.width + (4 if v else 3)
        g["res_bs"] = self.T * g["ldres"] + (4 if v else 1)
        g["col_off"] = 4 if v else 3
        g["ldo"] = g["col_off"] + self.width + (4 if v else 2)
        g["out_bs"] = self.T * g["ldo"] + (8 if v else 5)
        return g


# kind: ONE / SHORT / LONG; acc_cols 256 = two accumulators alternating over the tiles of a persistent CTA
CASES = [
    Case("t1_dense_cin4", 1, 1, 4, 128, plan=(ONE, 128, 1, 1)),
    Case("t127_k2_cin36_relu", 2, 127, 36, 80, taps=2, act=1, plan=(ONE, 128, 1, 2)),
    Case("t128_k16_long_one_wave", 3, 128, 128, 128, taps=16, act=1, affine=True, plan=(LONG, 128, 1, 3)),
    Case("t129_k5_tanh_affine_res", 4, 129, 80, 256, taps=5, act=3, affine=True, res=True, plan=(ONE, 128, 1, 0)),
    Case("t225_k4_affine_res", 2, 225, 128, 128, taps=4, affine=True, res=True, plan=(ONE, 128, 1, 4)),
    Case("t255_k7_sigmoid_scalar", 2, 255, 36, 80, taps=7, act=2, layout="scalar", plan=(ONE, 128, 0, 0)),
    Case("t257_k3_cin1024_relu_scalar", 2, 257, 1024, 256, taps=3, act=1, layout="scalar", plan=(LONG, 128, 0, 2)),
    Case("t1000_k8_cin4_cout768", 1, 1000, 4, 768, taps=8, act=1, plan=(ONE, 128, 1, 2)),
    Case("t37_dense_1025_scalar", 1, 37, 256, 1025, layout="scalar", plan=(ONE, 128, 0, 1)),
    Case("t300_k3_cin2048", 2, 300, 2048, 128, taps=3, act=1, affine=True, plan=(LONG, 128, 1, 3)),
    Case("t1000_n10_k3_cin1024_long_multi", 10, 1000, 1024, 256, taps=3, act=1, affine=True, plan=(LONG, 256, 1, 3)),
    Case("t1000_n8_dense_short_multi", 8, 1000, 128, 768, plan=(SHORT, 256, 1, 1)),
    Case("bank16_enc_n3", 3, 100, 128, 128, bank=16, act=1, affine=True, plan=(LONG, 128, 1, 3)),
    Case("bank16_enc_n32", 32, 100, 128, 128, bank=16, act=1, affine=True, plan=(LONG, 256, 1, 3)),
    Case("bank8_post_n2", 2, 129, 80, 128, bank=8, act=1, plan=(ONE, 128, 1, 2)),
    Case("bank8_post_scalar_n3", 3, 255, 80, 128, bank=8, act=1, affine=True, layout="scalar", plan=(ONE, 128, 0, 3)),
    # the config-3 shapes (batch 32, 1000 frames)
    Case("cfg3_final_dense_1025", 32, 1000, 256, 1025, layout="scalar", plan=(SHORT, 256, 0, 1)),
    Case("cfg3_post_proj1_3x1024_256", 32, 1000, 1024, 256, taps=3, act=1, affine=True, plan=(LONG, 256, 1, 3)),
    Case("cfg3_post_bank_8x128", 32, 1000, 80, 128, bank=8, act=1, affine=True, plan=(SHORT, 256, 1, 3)),
]
CASE_IDS = [c.name for c in CASES]


def plan_desc(c: Case, g=None):
    """taco_gemm_desc of a case with stand-in pointers (the plan reads only null-ness and 16-byte alignment)."""
    from tacotron_multispeaker_b200 import _abi
    g = g or c.geometry()
    d = _abi.TacoGemmDesc()
    d.N, d.T, d.Cin, d.Cout, d.taps, d.bank = c.N, c.T, c.Cin, c.Cout, c.taps, c.bank
    d.x, d.x_bs, d.ldx = FAKE, g["x_bs"], g["ldx"]
    d.w_host = FAKE
    d.bias_host = FAKE
    if c.affine:
        d.scale_host = d.shift_host = FAKE
    if c.res:
        d.res, d.res_bs, d.ldres = FAKE, g["res_bs"], g["ldres"]
    d.act = c.act
    d.out, d.out_bs, d.ldo, d.col_off = FAKE, g["out_bs"], g["ldo"], g["col_off"]
    return d


def kind_of(p):
    return ONE if not p["persistent"] else (LONG if p["long_k"] else SHORT)


def planned(c: Case, sms=SMS):
    from tacotron_multispeaker_b200 import _abi
    return _abi.umma_plan(plan_desc(c), sms)


# ---------------------------------------------------------------------------------------------------------------------
# host only: the launch plan
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    from tacotron_multispeaker_b200 import _abi
    from tacotron_multispeaker_b200.build import build_library
    build_library()
    return _abi.load()


@pytest.mark.parametrize("c", CASES, ids=CASE_IDS)
def test_case_plan(lib, c):
    p = planned(c)
    assert p["valid"] == 1
    assert (kind_of(p), p["acc_cols"], p["vec_epi"], p["variant"]) == c.plan, p
    assert p["acc_cols"] == (256 if p["ctas"] < p["tiles"] else 128)
    assert p["epi_warps"] == (4 if p["long_k"] else 8)
    taps = c.bank if c.bank > 1 else c.taps
    assert p["stages"] == (3 if p["long_k"] else 2 if p["persistent"] else (2 if taps * ((c.Cin + 63) // 64) >= 3 else 1))


def test_case_table_covers_every_plan_branch(lib):
    plans = [planned(c) for c in CASES]
    shapes = {(kind_of(p), p["acc_cols"]) for p in plans}
    # a short-K persistent launch has more than 2 x 148 tiles, hence always two accumulators
    assert shapes == {(ONE, 128), (SHORT, 256), (LONG, 128), (LONG, 256)}, shapes
    assert {p["variant"] for p in plans} == set(range(5))
    assert {p["vec_epi"] for p in plans} == {0, 1}
    assert {c.bank for c in CASES} == {1, 8, 16}
    assert {16, 8} <= {c.taps for c in CASES} and {1, 2, 3, 4, 5, 7} <= {c.taps for c in CASES}
    assert {4, 36, 80, 128, 1024, 2048} <= {c.Cin for c in CASES}
    assert {80, 128, 256, 768, 1025} <= {c.Cout for c in CASES}
    assert {1, 127, 128, 129, 255, 257, 1000} <= {c.T for c in CASES}
    assert any(97 <= c.T % 128 <= 104 for c in CASES)       # the last lane quarter of the last tile holds 1 .. 8 rows
    assert max(c.N for c in CASES) == 32 and min(c.N for c in CASES) == 1


def _cfg3(N=32, T=1000, **kw):
    return Case("", N, T, **kw)


# Every tensor-core GEMM of the config-3 forward (batch 32, 100 input symbols, 1000 output frames; the four highway layers
# run fused, see highway4 below) and the prenet at batch 1, against DESIGN.md "Launch shapes".
CONFIG3_LAUNCHES = [
    ("encoder prenet dense_1", _cfg3(T=100, Cin=320, Cout=256, act=1), (ONE, 128, 1, 2)),
    ("encoder prenet dense_2", _cfg3(T=100, Cin=256, Cout=128, act=1), (ONE, 128, 1, 2)),
    ("encoder prenet dense_1, batch 1", _cfg3(N=1, T=100, Cin=320, Cout=256, act=1), (ONE, 128, 1, 2)),
    ("encoder conv bank 16 x 128", _cfg3(T=100, Cin=128, Cout=128, bank=16, act=1, affine=True), (LONG, 256, 1, 3)),
    ("encoder proj_1 3 x 2048 -> 128", _cfg3(T=100, Cin=2048, Cout=128, taps=3, act=1, affine=True), (LONG, 128, 1, 3)),
    ("encoder proj_2", _cfg3(T=100, Cin=128, Cout=128, taps=3, affine=True, res=True), (ONE, 128, 1, 4)),
    ("encoder GRU input projection", _cfg3(T=100, Cin=128, Cout=768), (ONE, 128, 1, 1)),
    ("attention memory layer", _cfg3(T=100, Cin=256, Cout=256), (ONE, 128, 1, 1)),
    ("post-net conv bank 8 x 128", _cfg3(Cin=80, Cout=128, bank=8, act=1, affine=True), (SHORT, 256, 1, 3)),
    ("post-net proj_1 3 x 1024 -> 256", _cfg3(Cin=1024, Cout=256, taps=3, act=1, affine=True), (LONG, 256, 1, 3)),
    ("post-net proj_2", _cfg3(Cin=256, Cout=80, taps=3, affine=True, res=True), (ONE, 128, 1, 4)),
    ("post-net dense 80 -> 128", _cfg3(Cin=80, Cout=128), (ONE, 128, 1, 1)),
    ("post-net GRU input projection", _cfg3(Cin=128, Cout=768), (SHORT, 256, 1, 1)),
    ("final dense 256 -> 1025", _cfg3(Cin=256, Cout=1025), (SHORT, 256, 0, 1)),
]


@pytest.mark.parametrize("name,c,want", CONFIG3_LAUNCHES, ids=[n for n, _, _ in CONFIG3_LAUNCHES])
def test_config3_forward_plans(lib, name, c, want):
    from tacotron_multispeaker_b200 import _abi
    d = plan_desc(c)
    d.x_bs, d.ldx, d.col_off = c.T * c.Cin, c.Cin, 0          # the forward's dense tensors
    d.ldo = c.width
    d.out_bs = c.T * d.ldo
    if c.res:
        d.res_bs, d.ldres = c.T * c.Cout, c.Cout
    p = _abi.umma_plan(d, SMS)
    assert p["valid"] == 1 and (kind_of(p), p["acc_cols"], p["vec_epi"], p["variant"]) == want, p
    if name == "final dense 256 -> 1025":
        assert p["tiles"] == 2304 and p["epi_warps"] == 8 and p["stages"] == 2
    if name == "post-net proj_1 3 x 1024 -> 256":
        assert p["stages"] == 3 and p["epi_warps"] == 4 and p["ctas"] == SMS
    if name == "encoder prenet dense_1, batch 1":
        assert p["ctas"] == p["tiles"] == 2


def test_plan_refusals(lib):
    from tacotron_multispeaker_b200 import _abi
    c = Case("", 2, 50, 128, 80, act=1)
    ok = plan_desc(c)
    assert _abi.umma_plan(ok)["valid"] == 1
    for field, value in (("N", 0), ("Cin", 0), ("out", None)):
        d = plan_desc(c)
        setattr(d, field, value)
        assert _abi.umma_plan(d)["valid"] == 0, field
    d = plan_desc(c)
    d.scale_host = FAKE                                           # scale without shift
    assert _abi.umma_plan(d)["valid"] == 0
    d = plan_desc(c)
    d.col_off = 0
    d.out_hi = d.out_lo = FAKE
    d.out_cp = 128
    assert _abi.umma_plan(d)["valid"] == 1
    for field, value in (("out_cp", 64), ("out_cp", 96), ("out_cp", 256), ("col_off", 4), ("ldo", 81)):
        e = plan_desc(c)
        e.col_off = 0
        e.out_hi = e.out_lo = FAKE
        e.out_cp = 128
        setattr(e, field, value)
        assert _abi.umma_plan(e)["valid"] == 0, (field, value)


# ---------------------------------------------------------------------------------------------------------------------
# on the GPU: the arithmetic
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def eng(small_hp, small_weights):
    from tacotron_multispeaker_b200.engine import Engine
    e = Engine(small_hp, id_num=6)
    e.load_weights(small_weights)
    yield e
    e.set_gemm_mode(1)
    e.close()


def _filled32(n, dev="cuda"):
    return torch.full((n,), NAN32, dtype=torch.int32, device=dev).view(torch.float32)


def _filled16(n, dev="cuda"):
    return torch.full((n,), NAN16, dtype=torch.int16, device=dev).view(torch.bfloat16)


def _window_mask(N, T, width, col_off, ldo, out_bs, total):
    m = torch.zeros(total, dtype=torch.bool)
    torch.as_strided(m, (N, T, width), (out_bs, ldo, 1), col_off).fill_(True)
    return m


def _gather(buf, N, T, width, col_off, ldo, out_bs):
    return torch.as_strided(buf, (N, T, width), (out_bs, ldo, 1), col_off)


class Inputs:
    """Seeded fp32 inputs of a case, the strided device tensors and the float64 reference with its error scale."""

    def __init__(self, c: Case):
        rng = np.random.default_rng(zlib.crc32(c.name.encode()))
        self.c, g = c, c.geometry()
        self.g = g
        N, T, Cin, Cout = c.N, c.T, c.Cin, c.Cout
        self.x = rng.standard_normal((N, T, Cin)).astype(np.float32)
        nparam = Cout * c.bank
        taps = [ci + 1 for ci in range(c.bank)] if c.bank > 1 else [c.taps]
        self.ws = [(rng.standard_normal((k, Cin, Cout)) / np.sqrt(k * Cin)).astype(np.float32) for k in taps]
        self.b = (0.5 * rng.standard_normal(nparam)).astype(np.float32)
        self.scale = rng.uniform(-2, 2, nparam).astype(np.float32) if c.affine else None
        self.shift = rng.standard_normal(nparam).astype(np.float32) if c.affine else None
        self.r = rng.standard_normal((N, T, c.width)).astype(np.float32) if c.res else None
        self._ref = None

    def device(self):
        c, g = self.c, self.g
        xb = _filled32(c.N * g["x_bs"] + 16)
        _gather(xb, c.N, c.T, c.Cin, 0, g["ldx"], g["x_bs"]).copy_(torch.from_numpy(self.x))
        rb = None
        if c.res:
            rb = _filled32(c.N * g["res_bs"] + 16)
            _gather(rb, c.N, c.T, c.width, 0, g["ldres"], g["res_bs"]).copy_(torch.from_numpy(self.r))
        return xb, rb

    def reference(self):
        """(ref, tol scale S') in float64: ref = the operation; S' = sum |x||w| weighted as in the module docstring."""
        if self._ref is not None:
            return self._ref
        c = self.c
        x = torch.from_numpy(self.x).double()
        ax = x.abs()
        outs, Ss = [], []
        for w in self.ws:
            w = torch.from_numpy(w).double()
            zero = torch.zeros(w.shape[2], dtype=torch.float64)
            outs.append(O.conv1d_same(x, w, zero))
            Ss.append(O.conv1d_same(ax, w.abs(), zero))
        y = torch.cat(outs, -1) + torch.from_numpy(self.b).double()
        S = torch.cat(Ss, -1)
        y = [lambda v: v, torch.relu, torch.sigmoid, torch.tanh][c.act](y)
        rnd = y.abs()
        if c.affine:
            sc = torch.from_numpy(self.scale).double()
            y = y * sc + torch.from_numpy(self.shift).double()
            S = S * sc.abs().clamp(min=1.0)
            rnd = y.abs()
        if c.res:
            y = y + torch.from_numpy(self.r).double()
            rnd = rnd + y.abs()
        self._ref = (y, S, rnd)
        return self._ref

    def run(self, eng, out_split=None, write_out=True):
        """One taco_gemm_unit call in the engine's current mode; returns (plan, output buffer, x buffer)."""
        c, g = self.c, self.g
        xb, rb = self.device()
        total = (c.N + 1) * g["out_bs"]
        ob = _filled32(total) if write_out else None
        kw = dict(x=xb, x_bs=g["x_bs"], ldx=g["ldx"], taps=c.taps, bank=c.bank, act=c.act, bias=self.b, scale=self.scale,
                  shift=self.shift, out=ob, out_bs=g["out_bs"], ldo=g["ldo"], col_off=g["col_off"])
        if c.res:
            kw.update(res=rb, res_bs=g["res_bs"], ldres=g["ldres"])
        w = np.concatenate([a.reshape(-1) for a in self.ws])
        if out_split is not None:
            kw.update(out_split=out_split[:2], out_cp=out_split[2], col_off=0, ldo=c.width, out_bs=c.T * c.width)
        plan = eng.gemm_unit(c.N, c.T, c.Cin, c.Cout, w, **kw)
        torch.cuda.synchronize()
        return plan, ob, xb


def check_window(c, g, ob):
    """Outside the written window: the NaN pattern, bit for bit.  Inside: finite.  Returns the window [N, T, width]."""
    total = ob.numel()
    mask = _window_mask(c.N, c.T, c.width, g["col_off"], g["ldo"], g["out_bs"], total)
    bits = ob.view(torch.int32).cpu()
    outside = bits[~mask]
    assert bool((outside == NAN32).all()), "%d elements outside the window were written" % int((outside != NAN32).sum())
    win = _gather(ob.cpu(), c.N, c.T, c.width, g["col_off"], g["ldo"], g["out_bs"])
    assert bool(torch.isfinite(win).all()), "non-finite element inside the window"
    return win


def ratio(win, ref, S, rnd):
    """max over elements of (|got - ref| - C_ROUND rnd) / S: the smallest c for which got passes."""
    d = (win.double() - ref).abs() - C_ROUND * rnd
    return float((d / S.clamp(min=1e-30)).max())


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=CASE_IDS)
def test_gemm_against_fp64(eng, c):
    """Mode 1 within C_X3 of the fp64 reference, with the planned launch shape and nothing written outside the window; the
    same case in mode 2 must violate that bound (and meet C_BF16)."""
    I = Inputs(c)
    ref, S, rnd = I.reference()
    ratios = {}
    try:
        for mode in (1, 2):
            eng.set_gemm_mode(mode)
            plan, ob, _ = I.run(eng)
            if mode == 1:
                want = planned(c, torch.cuda.get_device_properties(0).multi_processor_count)
                assert plan == want, (plan, want)
            win = check_window(c, I.g, ob)
            ratios[mode] = ratio(win, ref, S, rnd)
            del ob, win
    finally:
        eng.set_gemm_mode(1)
    print("%s: worst |d| / S  mode 1 %.3e  mode 2 %.3e" % (c.name, ratios[1], ratios[2]))
    assert ratios[1] <= C_X3, ratios
    assert ratios[2] > C_X3, "a one-product run passes the bf16x3 bound: the bound cannot see a dropped correction product"
    assert ratios[2] <= C_BF16, ratios


def _bf16_split(v):
    hi = v.to(torch.bfloat16)
    lo = (v - hi.float()).to(torch.bfloat16)
    return hi, lo


COPY_CASES = [
    # (name, N, T, Cin, Cout, taps, act, affine, res, out_cp, consumer (taps, Cout))
    ("proj2_to_dense_80", 3, 129, 256, 80, 3, 0, True, True, 128, (1, 128)),
    ("prenet_relu_256", 2, 257, 320, 256, 1, 1, False, False, 256, (3, 128)),
    ("short_persistent_128", 38, 1000, 128, 128, 1, 1, True, False, 128, (16, 128)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("name,N,T,Cin,Cout,taps,act,affine,res,out_cp,consumer", COPY_CASES, ids=[c[0] for c in COPY_CASES])
def test_bf16_operand_copy(eng, name, N, T, Cin, Cout, taps, act, affine, res, out_cp, consumer):
    """The epilogue's bf16 hi / lo copy: hi == bf16_rne(out), lo == bf16_rne(out - hi) exactly (against a run of the same case
    with fp32 out; the copy-only run has out == NULL), padding channels Cout .. out_cp exactly zero, nothing written past
    the copy; a consumer GEMM reading the copy presplit equals, bit for bit, the same GEMM fed by a split pass of the fp32 out."""
    c = Case(name, N, T, Cin, Cout, taps=taps, act=act, affine=affine, res=res)
    I = Inputs(c)
    eng.set_gemm_mode(1)
    _, ob, _ = I.run(eng)
    out = check_window(c, I.g, ob)
    rows = N * T
    hi = _filled16(rows * out_cp + 64)
    lo = _filled16(rows * out_cp + 64)
    plan, none, _ = I.run(eng, out_split=(hi, lo, out_cp), write_out=False)
    assert none is None and plan["valid"] == 1 and plan["vec_epi"] == 1
    hic, loc = hi.view(torch.int16).cpu(), lo.view(torch.int16).cpu()
    assert bool((hic[rows * out_cp:] == NAN16).all()) and bool((loc[rows * out_cp:] == NAN16).all())
    H = hic[:rows * out_cp].view(N, T, out_cp)
    L = loc[:rows * out_cp].view(N, T, out_cp)
    eh, el = _bf16_split(out)
    assert torch.equal(H[..., :Cout], eh.view(torch.int16)), "hi != bf16_rne(out)"
    assert torch.equal(L[..., :Cout], el.view(torch.int16)), "lo != bf16_rne(out - hi)"
    assert bool((H[..., Cout:] == 0).all()) and bool((L[..., Cout:] == 0).all()), "padding channels are not zero"
    # consumer: presplit copy vs split pass of the fp32 output
    ktaps, kout = consumer
    rng = np.random.default_rng(5)
    w = (rng.standard_normal((ktaps, Cout, kout)) / np.sqrt(ktaps * Cout)).astype(np.float32)
    b = rng.standard_normal(kout).astype(np.float32)
    dense = out.contiguous().cuda()
    o1 = torch.empty(N, T, kout, device="cuda")
    o2 = torch.empty(N, T, kout, device="cuda")
    eng.gemm_unit(N, T, Cout, kout, w, x_split=(hi, lo), taps=ktaps, bias=b, act=1, out=o1)
    eng.gemm_unit(N, T, Cout, kout, w, x=dense, taps=ktaps, bias=b, act=1, out=o2)
    torch.cuda.synchronize()
    assert torch.equal(o1, o2)


# ---------------------------------------------------------------------------------------------------------------------
# highway4_kernel
# ---------------------------------------------------------------------------------------------------------------------
C_HW4 = 4e-6    # mode 1 bound of the layer chain: measured worst ratio 8.1e-7 (one row, one layer); mode 2 >= 1.4e-4
C_HW4_BF16 = 2.0 ** -6


def _hw_weights(layers, seed):
    rng = np.random.default_rng(seed)
    wh = (rng.standard_normal((layers, 128, 128)) / np.sqrt(128)).astype(np.float32)
    wt = (rng.standard_normal((layers, 128, 128)) / np.sqrt(128)).astype(np.float32)
    bh = (0.5 * rng.standard_normal((layers, 128))).astype(np.float32)
    bt = (0.5 * rng.standard_normal((layers, 128)) - 1.0).astype(np.float32)   # carry gate biased open as in training
    return wh, bh, wt, bt


def _hw_chain(x, wh, bh, wt, bt):
    """fp64 chain of highway layers and its error scale: per layer S_H + S_T |relu(H) - x| / 4, summed over the layers."""
    x = torch.from_numpy(x).double()
    S = torch.zeros_like(x)
    rnd = torch.zeros_like(x)
    for l in range(wh.shape[0]):
        Wh, Wt = torch.from_numpy(wh[l]).double(), torch.from_numpy(wt[l]).double()
        H = torch.relu(x @ Wh + torch.from_numpy(bh[l]).double())
        Tg = torch.sigmoid(x @ Wt + torch.from_numpy(bt[l]).double())
        S = S + x.abs() @ Wh.abs() + 0.25 * (x.abs() @ Wt.abs()) * (H - x).abs()
        y = H * Tg + x * (1 - Tg)
        rnd = rnd + y.abs() + x.abs()
        x = y
    return x, S, rnd


HW4_CASES = [
    # rows, layers, gemm mode, (fp32 out, bf16 copy)
    (1, 1, 1, (True, False)), (127, 2, 1, (True, True)), (128, 3, 2, (False, True)), (129, 4, 1, (True, True)),
    (18944, 4, 1, (True, False)), (18945, 3, 2, (True, True)), (32000, 4, 1, (True, True)), (32000, 2, 2, (True, False)),
    (129, 4, 2, (True, False)), (18945, 1, 1, (False, True)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("rows,layers,mode,outs", HW4_CASES, ids=["r%d-l%d-m%d-%s" % (r, l, m, "".join("oc"[i] for i in (0, 1) if o[i]))
                                                                  for r, l, m, o in HW4_CASES])
def test_highway4_against_fp64(eng, rows, layers, mode, outs):
    """The fused layers against the fp64 chain (bound C_HW4 in mode 1, C_HW4_BF16 in mode 2, and mode 2 must violate C_HW4),
    and the bf16 copy against bf16_rne(out) / bf16_rne(out - hi).  18944 = 148 x 128 rows: one tile per CTA; 18945 and
    32000 rows make CTAs walk two tiles.  Nothing is written past `rows`."""
    want_out, want_copy = outs
    wh, bh, wt, bt = _hw_weights(layers, rows + layers)
    x = np.random.default_rng(rows).standard_normal((rows, 128)).astype(np.float32)
    ref, S, rnd = _hw_chain(x, wh, bh, wt, bt)
    xd = torch.from_numpy(x).cuda()
    out = _filled32((rows + 1) * 128) if want_out else None
    hi = _filled16((rows + 1) * 128) if want_copy else None
    lo = _filled16((rows + 1) * 128) if want_copy else None
    eng.set_gemm_mode(mode)
    try:
        eng.highway4_unit(xd, wh, bh, wt, bt, out=out, out_split=(hi, lo) if want_copy else None)
        torch.cuda.synchronize()
    finally:
        eng.set_gemm_mode(1)
    c_mode = C_HW4 if mode == 1 else C_HW4_BF16
    tol = c_mode * S + C_ROUND * rnd
    if want_out:
        bits = out.view(torch.int32).cpu()
        assert bool((bits[rows * 128:] == NAN32).all())
        got = out[:rows * 128].view(rows, 128).cpu()
        assert bool(torch.isfinite(got).all())
        d = (got.double() - ref).abs()
        r = float(((d - C_ROUND * rnd) / S).max())
        print("highway4 rows=%d layers=%d mode %d: worst |d| / S = %.3e" % (rows, layers, mode, r))
        assert bool((d <= tol).all()), r
        if mode == 2:
            assert r > C_HW4, "a one-product run passes the bf16x3 bound"
    if want_copy:
        hic, loc = hi.view(torch.int16).cpu(), lo.view(torch.int16).cpu()
        assert bool((hic[rows * 128:] == NAN16).all()) and bool((loc[rows * 128:] == NAN16).all())
        H, L = hi[:rows * 128].view(rows, 128).cpu(), lo[:rows * 128].view(rows, 128).cpu()
        if want_out:
            eh, el = _bf16_split(got)
            assert torch.equal(H.view(torch.int16), eh.view(torch.int16))
            assert torch.equal(L.view(torch.int16), el.view(torch.int16))
        else:
            v = H.double() + L.double()
            assert bool(((v - ref).abs() <= tol + 2.0 ** -16 * ref.abs()).all())


@pytest.mark.gpu
def test_highway4_is_deterministic_under_repetition(eng):
    """32000 rows x 4 layers (each CTA walks two or more tiles), five runs: the fp32 output and the bf16 copy must be
    bit-identical.  Evidence against a data race in the kernel's shared-memory operand reuse, not a proof: a run cannot
    show that the write-after-read hazard between the second accumulator half's MMAs and the next operand write is gone
    (that fix is made from the code, and timing hid the hazard before it)."""
    rows = 32000
    wh, bh, wt, bt = _hw_weights(4, 99)
    xd = torch.from_numpy(np.random.default_rng(3).standard_normal((rows, 128)).astype(np.float32)).cuda()
    first = None
    for _ in range(5):
        out = torch.empty(rows, 128, device="cuda")
        hi = torch.empty(rows, 128, device="cuda", dtype=torch.bfloat16)
        lo = torch.empty(rows, 128, device="cuda", dtype=torch.bfloat16)
        eng.highway4_unit(xd, wh, bh, wt, bt, out=out, out_split=(hi, lo))
        torch.cuda.synchronize()
        cur = (out.clone(), hi.view(torch.int16).clone(), lo.view(torch.int16).clone())
        if first is None:
            first = cur
        else:
            for a, b in zip(cur, first):
                assert torch.equal(a, b)


# ---------------------------------------------------------------------------------------------------------------------
# host checks of the stage entry points: pointers and strides that would misalign the 16-byte vector loads are refused
# ---------------------------------------------------------------------------------------------------------------------
def _misaligned(shape):
    n = int(np.prod(shape))
    buf = torch.zeros(n + 1, device="cuda")
    v = buf[1:].view(*shape)            # contiguous, 4 bytes past a 16-byte boundary
    assert v.data_ptr() % 16 == 4
    return v


@pytest.mark.gpu
def test_stage_entry_points_refuse_misaligned_inputs(eng, small_hp):
    from tacotron_multispeaker_b200._abi import TacoError, TACO_ERR_INVALID
    N, T = 2, 9
    M = small_hp.num_mels
    calls = [
        ("cbhg", lambda: eng.cbhg(0, _misaligned((N, T, 128)))),
        ("postnet", lambda: eng.postnet(_misaligned((N, T, M)))),
        ("decode", lambda: eng.decode(_misaligned((N, T, 256)))),
        ("bigru", lambda: eng.bigru(0, _misaligned((N, T, 128)))),
        ("conv1d", lambda: eng.conv1d(_misaligned((N, T, 8)), np.ones((3, 8, 16), np.float32))),
    ]
    x = torch.zeros(N, T + 1, 128, device="cuda")
    mel = torch.zeros(N, T + 1, M, device="cuda")
    out = torch.empty(N, T, 256, device="cuda")
    lin = torch.empty(N, T, small_hp.num_freq, device="cuda")
    odd = (T * 128 + 1, T * M + 2)
    calls += [
        ("cbhg odd batch stride", lambda: eng._ck(eng.lib.taco_cbhg(eng._h, 0, C.c_void_p(x.data_ptr()), None, N, T, 0, odd[0],
                                                                    C.c_void_p(out.data_ptr()), eng.stream))),
        ("postnet odd batch stride", lambda: eng._ck(eng.lib.taco_postnet(eng._h, C.c_void_p(mel.data_ptr()), N, T, 0, odd[1],
                                                                          C.c_void_p(lin.data_ptr()), 0, eng.stream))),
    ]
    for name, call in calls:
        with pytest.raises(TacoError) as ei:
            call()
        assert ei.value.code == TACO_ERR_INVALID, name
    # the aligned calls still run
    eng.cbhg(0, x[:, :T].contiguous())
    eng.postnet(mel[:, :T].contiguous())
    torch.cuda.synchronize()
