"""Eight utterances per decoder cluster with the attention operands in tensor memory (DESIGN.md K7, layout TL_ATT).

At S = 8 the exp(2 key) rows and memory columns of a CTA do not fit shared memory next to the activation buffers; up to
T_in = 105 they live in tensor memory instead, and the weights they displace stream through the background warps' rings.  The
score and context phases keep the arithmetic and summation order of the shared-memory path, so S = 8 must give the same bits
as S = 5 for the same utterances.  Past the bound (T_in = 106) the non-resident path runs."""
import os

import numpy as np
import pytest
import torch

from conftest import make_inputs

pytestmark = pytest.mark.gpu

from oracle import taco_oracle as O  # noqa: E402

BOUND = 105   # largest T_in with the attention operands on chip at S = 8 (tests/test_decoder_plan.py pins it on the host)


@pytest.fixture(scope="module")
def eng(small_hp, small_weights):
    from tacotron_multispeaker_b200.engine import Engine
    e = Engine(small_hp, id_num=6)
    e.load_weights(small_weights)
    yield e
    e.close()


@pytest.fixture(scope="module")
def ow(small_weights):
    return O.W(small_weights, torch.float32)


def maxabs(a, b):
    return float((a.detach().cpu().double() - b.detach().cpu().double()).abs().max())


def _with_env(env, fn):
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return fn()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _case(eng, ow, hp, N, T_in, teacher, seed, S):
    rng = np.random.default_rng(seed)
    memory = (rng.standard_normal((N, T_in, 256)) * 0.5).astype(np.float32)
    targets = rng.uniform(0, 1, (N, hp.max_iters * hp.outputs_per_step, hp.num_mels)).astype(np.float32)
    dec, al, steps = _with_env({"TACO_DEC_S": S}, lambda: eng.decode(memory, targets if teacher else None, teacher))
    rdec, ral, rsteps = O.decode(torch.from_numpy(memory), ow, hp.num_mels, hp.outputs_per_step, hp.max_iters,
                                 torch.from_numpy(targets) if teacher else None, teacher)
    assert steps == rsteps
    return maxabs(dec, rdec), maxabs(al, ral), al, ral


@pytest.mark.parametrize("T_in", [37, 60, 100, BOUND, BOUND + 1])
def test_eight_per_cluster_against_oracle(eng, ow, small_hp, T_in):
    """S = 8 (two clusters of eight) at lengths inside and just past the tensor-memory bound, teacher forced and free running,
    with the bounds of the other decoder tests."""
    e_dec, e_al, al, ral = _case(eng, ow, small_hp, 16, T_in, True, 300 + T_in, 8)
    assert e_dec < 2e-4 and e_al < 1e-5
    assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))
    e_dec, e_al, _, _ = _case(eng, ow, small_hp, 16, T_in, False, 400 + T_in, 8)
    assert e_dec < 1e-3 and e_al < 1e-4


def test_eight_per_cluster_exact_softmax(small_hp, small_weights):
    """||v||_1 > 40: raw scores and the row maximum (the true softmax) with the operands in tensor memory."""
    from tacotron_multispeaker_b200.engine import Engine
    w = dict(small_weights)
    vname = [k for k in w if k.endswith("bahdanau_attention/attention_v")][0]
    mname = [k for k in w if k.endswith("memory_layer/kernel")][0]
    w[vname] = (w[vname] * 25.0).astype(np.float32)
    w[mname] = (w[mname] * 3.0).astype(np.float32)
    assert np.abs(w[vname]).sum() > 100.0
    e = Engine(small_hp, id_num=6)
    try:
        e.load_weights(w)
        wo = O.W(w, torch.float32)
        for teacher in (True, False):
            e_dec, e_al, al, ral = _case(e, wo, small_hp, 8, 80, teacher, 33, 8)
            assert e_dec < (2e-4 if teacher else 1e-3), (teacher, e_dec)
            assert e_al < (1e-4 if teacher else 1e-3), (teacher, e_al)
            assert float(ral.max()) > 0.5
            if teacher:
                assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))
    finally:
        e.close()


@pytest.mark.parametrize("teacher", [False, True])
def test_eight_and_five_per_cluster_bit_identical(teacher):
    """Config 3 (batch 32, T_in 100, r = 5): S = 8 (tensor memory) and S = 5 (shared memory) give the same bits."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    e = Engine(hp, 60)
    try:
        e.load_weights(random_init(hp, 60, seed=1234))
        rng = np.random.default_rng(8)
        memory = torch.from_numpy((rng.standard_normal((32, 100, 256)) * 0.5).astype(np.float32)).cuda()
        tg = torch.from_numpy(rng.uniform(0, 1, (32, 1000, 80)).astype(np.float32)).cuda() if teacher else None
        d5, a5, s5 = _with_env({"TACO_DEC_S": 5}, lambda: e.decode(memory, tg, teacher))
        d8, a8, s8 = _with_env({"TACO_DEC_S": 8}, lambda: e.decode(memory, tg, teacher))
    finally:
        e.close()
    assert s5 == s8
    assert torch.equal(d5, d8) and torch.equal(a5, a8)


def _config3_forward(e, seed):
    ids, lengths, spk = make_inputs(32, 100, 60, seed, min_len=60, vocab=(7108, 7325))
    mel, lin, al, steps = e.forward(ids, lengths, spk)
    torch.cuda.synchronize()
    return mel.clone(), lin.clone(), al.clone(), steps


def test_config3_default_geometry_matches_seven_clusters():
    """A full-size config-3 forward in the default geometry (4 clusters of 8) is bit-identical to 7 clusters of 5 / 4."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    e = Engine(hp, 60)
    try:
        e.load_weights(random_init(hp, 60, seed=1234))
        geo = e.decoder_geometry(32)
        assert (geo["num_clusters"], geo["samples_per_cluster"]) == (4, 8)
        got = _config3_forward(e, 1)
        ref = _with_env({"TACO_DEC_NCL": 7}, lambda: _config3_forward(e, 1))
    finally:
        e.close()
    assert got[3] == ref[3]
    for a_, b_ in zip(got[:3], ref[:3]):
        assert torch.equal(a_, b_)


def test_eight_per_cluster_deterministic_under_repetition():
    """Twelve config-3 forwards in the default geometry (4 clusters of 8, operands in tensor memory, the longer weight rings)
    are bit-identical while a second handle keeps the other SMs busy on another stream."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    w = random_init(hp, 60, seed=1234)
    e = Engine(hp, 60); e.load_weights(w)
    noise = Engine(hp, 60); noise.load_weights(w)
    side = torch.cuda.Stream(device=torch.device("cuda", 0))
    try:
        ids, lengths, spk = make_inputs(32, 100, 60, 39, min_len=50, vocab=(7108, 7325))
        nids, nlen, nspk = make_inputs(8, 50, 60, 3, min_len=30, vocab=(7108, 7325))
        first = None
        for rep in range(12):
            with torch.cuda.stream(side):
                noise.forward(nids, nlen, nspk)
            mel, lin, al, steps = e.forward(ids, lengths, spk)
            torch.cuda.synchronize()
            cur = (mel.clone(), lin.clone(), al.clone())
            if first is None:
                first = cur
            else:
                for a_, b_ in zip(cur, first):
                    assert torch.equal(a_, b_), "run %d differs from run 0" % rep
    finally:
        e.close(); noise.close()
