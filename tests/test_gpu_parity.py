"""Parity of the CUDA path (through the C ABI) against the CPU oracle.

Tolerances (fp32 mode): stage outputs 2e-4 max-abs, whole teacher-forced
forward 1e-3 max-abs on mel / linear (north_star), alignments 1e-4.
Free-running decodes feed rounding differences back through the loop, so they
get a looser bound and the exact properties instead (step count, shapes).
"""
import os

import numpy as np
import pytest
import torch

from conftest import make_inputs

pytestmark = pytest.mark.gpu

from oracle import taco_oracle as O  # noqa: E402  (tests may use the oracle)


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
    a = a.detach().cpu().double() if isinstance(a, torch.Tensor) else torch.as_tensor(a).double()
    b = b.detach().cpu().double() if isinstance(b, torch.Tensor) else torch.as_tensor(b).double()
    assert a.shape == b.shape, (a.shape, b.shape)
    return float((a - b).abs().max())


def test_library_loaded_is_in_tree():
    from tacotron_multispeaker_b200 import _abi
    lib = _abi.load()
    assert os.path.dirname(_abi.LIB_PATH).endswith("tacotron_multispeaker_b200")
    assert b"sm_100a" in lib.taco_version()


def test_weight_inventory_matches_python(eng, small_hp):
    from tacotron_multispeaker_b200.weights import weight_specs
    assert sorted(eng.weight_names()) == sorted(weight_specs(small_hp, 6).keys())


def test_embed(eng, ow):
    ids, lengths, spk = make_inputs(5, 13, 6, 0)
    got = eng.embed(ids, spk)
    ref = O.embed(ids, spk, ow)
    assert maxabs(got, ref) == 0.0          # pure gather: bit exact
    eng.check_ids()


def test_embed_oob_id_flags_error(eng):
    from tacotron_multispeaker_b200._abi import TacoError, TACO_ERR_OOB_ID
    ids, lengths, spk = make_inputs(2, 5, 6, 1)
    ids[1, 2] = 7352 + 5
    out = eng.embed(ids, spk)
    with pytest.raises(TacoError) as ei:
        eng.check_ids()
    assert ei.value.code == TACO_ERR_OOB_ID
    assert float(out[1, 2, :256].abs().max()) == 0.0   # zero row, like TF GPU gather
    eng.check_ids()                                    # flag is cleared


@pytest.mark.parametrize("k,cin,cout,act", [(1, 128, 128, 1), (2, 80, 128, 1), (3, 256, 80, 0),
                                            (4, 128, 128, 1), (7, 80, 128, 3), (16, 128, 128, 1),
                                            (1, 256, 1025, 0), (3, 2048, 128, 2), (1, 320, 256, 1)])
@pytest.mark.parametrize("mode,tol", [(1, 1e-4), (2, 6e-2)])
def test_conv1d_same(eng, k, cin, cout, act, mode, tol):
    """tf.layers.conv1d('same') + bias + activation.  mode 1 = tcgen05 with bf16 hi/lo split operands
    (default; fp32-class), 2 = plain bf16 tcgen05 (stated looser tolerance)."""
    rng = np.random.default_rng(k * 1000 + cin + cout)
    N, T = 3, 37
    x = rng.standard_normal((N, T, cin)).astype(np.float32)
    w = (rng.standard_normal((k, cin, cout)) / np.sqrt(k * cin)).astype(np.float32)
    b = rng.standard_normal((cout,)).astype(np.float32)
    eng.set_gemm_mode(mode)
    try:
        got = eng.conv1d(x, w, b, act)
    finally:
        eng.set_gemm_mode(1)
    ref = O.conv1d_same(torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b))
    ref = [lambda v: v, torch.relu, torch.sigmoid, torch.tanh][act](ref)
    assert maxabs(got, ref) < tol


def test_conv1d_even_kernel_padding_kat(eng):
    # unit impulse, distinct taps: 'same' pads (k-1)//2 on the left (SURVEY 8c KAT 4)
    k, T = 4, 9
    x = np.zeros((1, T, 4), np.float32)
    x[0, 4, 0] = 1.0
    w = np.zeros((k, 4, 4), np.float32)
    for j in range(k):
        w[j, 0, 0] = j + 1
    got = eng.conv1d(x, w, None, 0)[0, :, 0].cpu().numpy()   # small integers are exact in bf16 too
    exp = np.zeros(T, np.float32)
    for j in range(k):           # y[t] = sum_j x[t + j - 1] w[j]  -> impulse at t = 4 - j + 1
        exp[4 - j + 1] = j + 1
    assert np.array_equal(got, exp)


@pytest.mark.parametrize("N,T,C,affine", [(1, 1, 4, False), (2, 7, 128, True), (3, 100, 2048, True), (5, 33, 1024, False)])
def test_maxpool_affine_kat(eng, N, T, C, affine):
    """a5 in isolation: max_pooling1d(2, 1, 'same') after the folded BN affine (modules.py:45-49): out[t] = max(a(x[t]), a(x[t+1])),
    the last row passes through.  Bit exact against the oracle (max and one FMA per element)."""
    rng = np.random.default_rng(N * 1000 + T)
    x = rng.standard_normal((N, T, C)).astype(np.float32)
    sc = rng.uniform(-2, 2, C).astype(np.float32) if affine else None       # negative scales: the affine must come BEFORE the max
    sh = rng.standard_normal(C).astype(np.float32) if affine else None
    got = eng.maxpool_affine(x, sc, sh).cpu()
    xa = torch.from_numpy(x)
    if affine:
        xa = torch.addcmul(torch.from_numpy(sh), xa, torch.from_numpy(sc))   # fused multiply-add like the kernel
    ref = O.max_pool_same2(xa)
    assert maxabs(got, ref) < 1e-6
    assert torch.equal(got[:, -1], xa[:, -1])


@pytest.mark.parametrize("N,T,C", [(1, 2, 4), (3, 50, 128), (32, 100, 2048), (2, 1000, 256)])
def test_bn_batch_stats_kat(eng, N, T, C):
    """Training-mode batch normalisation in isolation (modules.py:101 with is_training): biased moments over (N, T) accumulated in
    double, folded into scale / shift with epsilon 1e-3; scale * x + shift must equal the oracle's batch_norm(mode='batch')."""
    rng = np.random.default_rng(C + T)
    x = (rng.standard_normal((N, T, C)) * rng.uniform(0.1, 3.0, C) + rng.standard_normal(C)).astype(np.float32)
    gamma = rng.uniform(0.5, 2.0, C).astype(np.float32)
    beta = rng.standard_normal(C).astype(np.float32)
    scale, shift = eng.bn_batch_stats(x, gamma, beta)
    xt = torch.from_numpy(x)
    got = xt * scale.cpu() + shift.cpu()
    ref = O.batch_norm(xt.double(), torch.from_numpy(gamma).double(), torch.from_numpy(beta).double(), None, None, "batch")
    assert maxabs(got, ref) < 2e-5
    var = xt.double().var(dim=(0, 1), unbiased=False)
    want = torch.from_numpy(gamma).double() / torch.sqrt(var + 1e-3)
    assert float(((scale.cpu().double() - want).abs() / want.abs()).max()) < 1e-5


@pytest.mark.parametrize("which,N,T,masked", [(0, 5, 23, True), (0, 3, 11, False), (1, 2, 60, False),
                                              (0, 80, 9, True), (1, 1, 150, False), (0, 8, 31, True), (0, 9, 31, True), (1, 33, 40, False),
                                              (0, 149, 40, True)])
def test_bigru(eng, ow, which, N, T, masked):
    rng = np.random.default_rng(N * 100 + T)
    x = rng.standard_normal((N, T, 128)).astype(np.float32)
    lengths = None
    if masked:
        lengths = rng.integers(1, T + 1, (N,)).astype(np.int32)
        lengths[0] = T
    got = eng.bigru(which, x, lengths)
    ref = O.bigru(torch.from_numpy(x), lengths, ow, "encoder_cbhg" if which == 0 else "post_cbhg")
    assert maxabs(got, ref) < 1e-4
    if masked:   # outputs exactly zero beyond each length (KAT 7)
        g = got.cpu().numpy()
        for i in range(N):
            assert np.all(g[i, lengths[i]:] == 0.0)


@pytest.mark.parametrize("which,N,T,masked", [(0, 5, 23, True), (1, 2, 60, False), (0, 19, 9, True), (1, 8, 40, True),
                                              (0, 16, 31, True)])
def test_bigru_tensor_core_variant(eng, ow, which, N, T, masked, monkeypatch):
    """TACO_BIGRU=mma: the same recurrence on mma.sync with the recurrent weights in tensor memory, 8 utterances per
    CTA (bf16 hi/lo operands: fp32-class; ragged lengths, a last CTA with fewer than 8 utterances)."""
    monkeypatch.setenv("TACO_BIGRU", "mma")
    rng = np.random.default_rng(N * 100 + T)
    x = rng.standard_normal((N, T, 128)).astype(np.float32)
    lengths = None
    if masked:
        lengths = rng.integers(1, T + 1, (N,)).astype(np.int32)
        lengths[0] = T
    got = eng.bigru(which, x, lengths)
    ref = O.bigru(torch.from_numpy(x), lengths, ow, "encoder_cbhg" if which == 0 else "post_cbhg")
    assert maxabs(got, ref) < 2e-4


@pytest.mark.parametrize("which,bn", [(0, "moving"), (0, "batch"), (1, "moving"), (1, "batch")])
def test_cbhg(eng, ow, which, bn):
    rng = np.random.default_rng(which * 10 + len(bn))
    N, T = 3, 29
    cin = 128 if which == 0 else 80
    x = rng.standard_normal((N, T, cin)).astype(np.float32)
    lengths = np.array([29, 17, 5], np.int32) if which == 0 else None
    got = eng.cbhg(which, x, lengths, 1 if bn == "batch" else 0)
    ref = O.cbhg(torch.from_numpy(x), lengths, ow, "encoder_cbhg" if which == 0 else "post_cbhg",
                 16 if which == 0 else 8, bn)
    assert maxabs(got, ref) < 2e-4


def test_encoder(eng, ow):
    ids, lengths, spk = make_inputs(4, 21, 6, 3)
    got = eng.encoder(ids, lengths, spk, 0)
    ref = O.encoder(ids, lengths, spk, ow, "moving")
    assert maxabs(got, ref) < 2e-4


def _decode_case(eng, ow, hp, N, T_in, teacher, seed, S=None):
    rng = np.random.default_rng(seed)
    memory = (rng.standard_normal((N, T_in, 256)) * 0.5).astype(np.float32)
    targets = rng.uniform(0, 1, (N, hp.max_iters * hp.outputs_per_step, hp.num_mels)).astype(np.float32)
    if S is not None:
        os.environ["TACO_DEC_S"] = str(S)
    try:
        dec, al, steps = eng.decode(memory, targets if teacher else None, teacher)
    finally:
        os.environ.pop("TACO_DEC_S", None)
    rdec, ral, rsteps = O.decode(torch.from_numpy(memory), ow, hp.num_mels, hp.outputs_per_step, hp.max_iters,
                                 torch.from_numpy(targets) if teacher else None, teacher)
    assert steps == rsteps
    return maxabs(dec, rdec), maxabs(al, ral), al, ral


@pytest.mark.parametrize("N,T_in,S", [(1, 7, None), (3, 19, None), (5, 33, 2), (8, 16, 4), (9, 50, 8),
                                      (17, 100, None), (2, 130, 1)])
def test_decode_teacher_forced(eng, ow, small_hp, N, T_in, S):
    e_dec, e_al, al, ral = _decode_case(eng, ow, small_hp, N, T_in, True, N * 7 + T_in, S)
    assert e_dec < 2e-4 and e_al < 1e-5
    # identical per-step attention argmax (north_star)
    assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))


@pytest.mark.parametrize("N,T_in", [(1, 1), (2, 2), (1, 512), (3, 511), (70, 9), (2, 300)])
def test_decode_extreme_shapes(eng, ow, small_hp, N, T_in):
    """Edges of the decoder's geometry: a single input position (softmax over one key), the largest supported T_in (512:
    attention operands no longer resident in shared memory), more utterances than one wave of clusters holds (70 -> 9 clusters
    of 8 in two waves), odd lengths around the 16-range pair cut.  Teacher forced and free running against the oracle."""
    e_dec, e_al, al, ral = _decode_case(eng, ow, small_hp, N, T_in, True, 31 * N + T_in)
    assert e_dec < 2e-4 and e_al < 1e-5
    assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))
    e_dec, e_al, _, _ = _decode_case(eng, ow, small_hp, N, T_in, False, 17 * N + T_in)
    assert e_dec < 1e-3 and e_al < 1e-4


def test_decode_rejects_longer_inputs(eng, small_hp):
    """T_in > 512 is refused loudly (TACO_ERR_UNSUPPORTED), not truncated."""
    mem = np.zeros((1, 513, 256), np.float32)
    with pytest.raises(RuntimeError):
        eng.decode(mem, None, False)


@pytest.mark.parametrize("N,T_in", [(1, 1), (2, 3), (40, 5)])
def test_forward_ragged_and_tiny_batches(eng, ow, small_hp, small_weights, N, T_in):
    """Whole path on the smallest inputs the reference's feeder can produce: one symbol, lengths of 1 inside a padded batch (the
    BiGRU masks everything but the first step), a batch larger than 32."""
    ids, lengths, spk = make_inputs(N, T_in, 6, 3 * N + T_in, min_len=1)
    lengths[-1] = 1
    ids[-1, 1:] = 0
    mel, lin, al, steps = eng.forward(ids, lengths, spk)
    ref = O.tacotron_forward(small_weights, small_hp, ids, lengths, identities=spk, id_num=6)
    assert steps == ref["steps"]
    assert maxabs(mel, ref["mel_outputs"]) < 1e-3 and maxabs(lin, ref["linear_outputs"]) < 1e-3
    assert maxabs(al, ref["alignments"]) < 1e-4


def test_utterances_are_independent(eng, small_hp):
    """Moving-statistics synthesis treats the utterances of a batch independently (no op of the graph mixes batch entries): a
    batch of six equals six batches of one.  The two runs take different decoder paths (clusters of several utterances with
    all-warp attention vs one utterance per cluster with critical-group attention), so this also ties those together."""
    ids, lengths, spk = make_inputs(6, 23, 6, 77)
    mel, lin, al, steps = eng.forward(ids, lengths, spk)
    for i in range(6):
        m1, l1, a1, s1 = eng.forward(ids[i:i + 1], lengths[i:i + 1], spk[i:i + 1])
        assert s1 == steps
        assert maxabs(m1, mel[i:i + 1]) < 1e-4 and maxabs(l1, lin[i:i + 1]) < 1e-4 and maxabs(a1, al[i:i + 1]) < 1e-5


def test_teacher_forcing_with_own_outputs_reproduces_free_run(eng, small_hp):
    """TacoTrainingHelper fed with the model's own frames must walk the same trajectory as TacoTestHelper (helpers.py:26-38 vs
    68-77).  On the device the two take different arithmetic: the free run never forms the fed-back frame (the output projection
    is folded into the prenet's first layer in double precision), teacher forcing reads the frame from memory."""
    ids, lengths, spk = make_inputs(4, 21, 6, 5)
    mel, lin, al, steps = eng.forward(ids, lengths, spk)
    mel2, lin2, al2, steps2 = eng.forward(ids, lengths, spk, mel_targets=mel.contiguous(), teacher_force=True, bn_mode=0)
    assert steps2 == steps
    assert maxabs(mel2, mel) < 1e-4 and maxabs(lin2, lin) < 1e-4 and maxabs(al2, al) < 1e-5


@pytest.mark.parametrize("seed", list(range(10)))
def test_forward_random_configs(seed):
    """Seeded sweep over hyper-parameters the fixed cases do not reach: r in 1..6 (output projection of 80 r columns cut into
    16-column tiles over the cluster), odd max_iters, odd T_in, speaker tables of different sizes and the single-speaker branch,
    batch sizes that cut unevenly into clusters; free running, teacher forced with moving statistics and with batch statistics."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    rng = np.random.default_rng(1000 + seed)
    r = int(rng.integers(1, 7))
    iters = int(rng.integers(2, 8))
    N = int(rng.integers(1, 14))
    T_in = int(rng.integers(1, 70))
    id_num = int(rng.choice([0, 2, 7, 400]))
    mode = ("free", "teacher_moving", "teacher_batch")[seed % 3]
    hp = HParams(outputs_per_step=r, max_iters=iters)
    w = random_init(hp, id_num, seed=seed, randomize_bn=True)
    ids, lengths, spk = make_inputs(N, T_in, max(id_num, 1), seed, min_len=1)
    spk_arg = spk if id_num > 1 else None
    e = Engine(hp, id_num)
    try:
        e.load_weights(w)
        if mode == "free":
            mel, lin, al, steps = e.forward(ids, lengths, spk_arg)
            ref = O.tacotron_forward(w, hp, ids, lengths, identities=spk_arg, id_num=id_num)
        else:
            T_tgt = int(rng.integers(r, iters * r + 3))
            tg = rng.uniform(0, 1, (N, T_tgt, hp.num_mels)).astype(np.float32)
            bn = "batch" if mode == "teacher_batch" else "moving"
            mel, lin, al, steps = e.forward(ids, lengths, spk_arg, tg, True, 1 if bn == "batch" else 0)
            ref = O.tacotron_forward(w, hp, ids, lengths, mel_targets=tg, identities=spk_arg, id_num=id_num, teacher_force=True, bn_mode=bn)
    finally:
        e.close()
    assert steps == ref["steps"], (r, iters, N, T_in, id_num, mode)
    assert maxabs(mel, ref["mel_outputs"]) < 1e-3, (r, iters, N, T_in, id_num, mode)
    assert maxabs(lin, ref["linear_outputs"]) < 1e-3, (r, iters, N, T_in, id_num, mode)
    assert maxabs(al, ref["alignments"]) < 1e-4, (r, iters, N, T_in, id_num, mode)


def test_ffma_decoder_fallback(monkeypatch, small_weights, small_hp):
    """The fp32 FFMA cluster decoder (csrc/decoder.cu) ships as the fallback for shapes the tensor-core decoder does not take
    (num_mels not a multiple of 16, or more than 128) and behind TACO_DEC_IMPL=v2: same bounds as the default decoder."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    # (a) forced by the developer switch, standard hyper-parameters
    monkeypatch.setenv("TACO_DEC_IMPL", "v2")
    e = Engine(small_hp, 6)
    try:
        e.load_weights(small_weights)
        wo = O.W(small_weights, torch.float32)
        for N, T_in, teacher in ((3, 19, True), (9, 50, True), (4, 25, False)):
            e_dec, e_al, al, ral = _decode_case(e, wo, small_hp, N, T_in, teacher, 5 * N + T_in)
            assert e_dec < (2e-4 if teacher else 1e-3) and e_al < (1e-5 if teacher else 1e-4)
    finally:
        e.close()
    monkeypatch.delenv("TACO_DEC_IMPL")
    # (b) taken automatically: 72 mel channels (4.5 tiles of 16) -- whole path against the oracle
    hp = HParams(outputs_per_step=3, max_iters=5, num_mels=72)
    w = random_init(hp, 4, seed=9, randomize_bn=True)
    ids, lengths, spk = make_inputs(3, 17, 4, 2)
    e = Engine(hp, 4)
    try:
        e.load_weights(w)
        mel, lin, al, steps = e.forward(ids, lengths, spk)
        ref = O.tacotron_forward(w, hp, ids, lengths, identities=spk, id_num=4)
        assert steps == ref["steps"]
        assert maxabs(mel, ref["mel_outputs"]) < 1e-3 and maxabs(lin, ref["linear_outputs"]) < 1e-3
        assert maxabs(al, ref["alignments"]) < 1e-4
    finally:
        e.close()


@pytest.mark.parametrize("N,T_in", [(3, 19), (17, 100)])
def test_decode_bf16_mode(eng, ow, small_hp, N, T_in):
    """taco_set_gemm_mode(2): the decoder multiplies W_hi x_hi only (plain bf16 operands, fp32 accumulation, one MMA per
    chunk-tile instead of three).  Stated tolerance of the decoder in this mode: 1e-2 max-abs on its outputs, 1e-3 on the
    alignments (measured 2.7e-3 / 1.7e-4; the fp32-class default meets 2e-4 / 1e-5 on the same cases).  At full size (32 x 1000
    frames, free running) the mode differs from the default by 4.4e-3 on mel and 1.4e-3 on linear."""
    eng.set_gemm_mode(2)
    try:
        e_dec, e_al, al, ral = _decode_case(eng, ow, small_hp, N, T_in, True, N * 7 + T_in, None)
        e_dec_f, e_al_f, _, _ = _decode_case(eng, ow, small_hp, N, T_in, False, N * 7 + T_in, None)
    finally:
        eng.set_gemm_mode(1)
    print("bf16 decoder mode: teacher-forced %.2e / %.2e, free-running %.2e / %.2e" % (e_dec, e_al, e_dec_f, e_al_f))
    assert e_dec < 1e-2 and e_al < 1e-3
    assert e_dec_f < 1e-2 and e_al_f < 1e-3
    assert e_dec > 1e-5          # the mode really is coarser than the default: it ran the one-product kernel


@pytest.mark.parametrize("N,T_in,S", [(1, 11, None), (4, 25, None), (6, 40, 4)])
def test_decode_free_running(eng, ow, small_hp, N, T_in, S):
    e_dec, e_al, _, _ = _decode_case(eng, ow, small_hp, N, T_in, False, N * 11 + T_in, S)
    assert e_dec < 1e-3 and e_al < 1e-4


@pytest.mark.parametrize("scale,N,T_in,tol_al", [(10.0, 3, 29, 1e-5), (25.0, 6, 50, 1e-4)])   # scores of +-350 carry ~4e-5 of fp32 rounding into exp()
def test_decode_large_attention_v(small_hp, small_weights, scale, N, T_in, tol_al):
    """A trained checkpoint can have ||attention_v||_1 far above the 40 for which exp(score - ||v||_1) is safe in fp32: the decoder
    then exchanges raw scores and subtracts the row maximum (a true softmax, reference BahdanauAttention).  Random-init v has
    ||v||_1 ~ 14, so scale it (and the keys through the memory layer) until scores spread over +-100."""
    from tacotron_multispeaker_b200.engine import Engine
    w = dict(small_weights)
    vname = [k for k in w if k.endswith("bahdanau_attention/attention_v")][0]
    mname = [k for k in w if k.endswith("memory_layer/kernel")][0]
    w[vname] = (w[vname] * scale).astype(np.float32)
    w[mname] = (w[mname] * 3.0).astype(np.float32)
    assert np.abs(w[vname]).sum() > 100.0
    e = Engine(small_hp, id_num=6)
    try:
        e.load_weights(w)
        wo = O.W(w, torch.float32)
        for teacher in (True, False):
            e_dec, e_al, al, ral = _decode_case(e, wo, small_hp, N, T_in, teacher, int(scale) + N)
            assert e_dec < (2e-4 if teacher else 1e-3), (teacher, e_dec)
            assert e_al < (tol_al if teacher else 10 * tol_al), (teacher, e_al)
            assert float(ral.max()) > 0.5          # the attention is sharply peaked: rows far below the maximum must underflow to 0, not to a floor
            if teacher:
                assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))
    finally:
        e.close()


def test_postnet(eng, ow, small_hp):
    rng = np.random.default_rng(5)
    mel = rng.uniform(-0.5, 1.0, (2, 35, 80)).astype(np.float32)
    got = eng.postnet(mel, 0)
    post = O.cbhg(torch.from_numpy(mel), None, ow, "post_cbhg", 8, "moving")
    ref = O.dense(post, ow("dense/kernel"), ow("dense/bias"))
    assert maxabs(got, ref) < 2e-4


@pytest.mark.parametrize("mode", ["free", "teacher_moving", "teacher_batch"])
def test_forward_whole_path(eng, small_hp, small_weights, mode):
    hp = small_hp
    N, T_in = 4, 24
    ids, lengths, spk = make_inputs(N, T_in, 6, 11)
    rng = np.random.default_rng(2)
    T_out = hp.max_iters * hp.outputs_per_step
    mel_t = rng.uniform(0, 1, (N, T_out, hp.num_mels)).astype(np.float32)
    lin_t = np.zeros((N, T_out, hp.num_freq), np.float32)
    if mode == "free":
        ref = O.tacotron_forward(small_weights, hp, ids, lengths, identities=spk, id_num=6)
        mel, lin, al, steps = eng.forward(ids, lengths, spk)
        tol = 1e-3
    elif mode == "teacher_moving":
        ref = O.tacotron_forward(small_weights, hp, ids, lengths, mel_targets=mel_t, identities=spk, id_num=6,
                                 teacher_force=True, bn_mode="moving")
        mel, lin, al, steps = eng.forward(ids, lengths, spk, mel_t, True, 0)
        tol = 1e-3
    else:   # reference-faithful training forward: teacher forcing + batch-statistics BN
        ref = O.tacotron_forward(small_weights, hp, ids, lengths, mel_targets=mel_t, linear_targets=lin_t,
                                 identities=spk, id_num=6)
        mel, lin, al, steps = eng.forward(ids, lengths, spk, mel_t, True, 1)
        tol = 1e-3
    assert steps == ref["steps"]
    assert maxabs(mel, ref["mel_outputs"]) < tol
    assert maxabs(lin, ref["linear_outputs"]) < tol
    assert maxabs(al, ref["alignments"]) < 1e-4
    if mode != "free":
        assert torch.equal(al.cpu().argmax(dim=1), ref["alignments"].argmax(dim=1))


@pytest.mark.parametrize("mode,tol", [(2, 5e-2)])
def test_forward_other_gemm_modes(eng, small_hp, small_weights, mode, tol):
    """Plain-bf16 tensor-core mode meets the stated looser tolerance (5e-2 max-abs on mel/linear, teacher-forced).  Modes
    other than 1 and 2 are refused."""
    from tacotron_multispeaker_b200._abi import TacoError, TACO_ERR_INVALID
    with pytest.raises(TacoError) as ei:
        eng.set_gemm_mode(0)
    assert ei.value.code == TACO_ERR_INVALID
    hp = small_hp
    ids, lengths, spk = make_inputs(3, 20, 6, 13)
    rng = np.random.default_rng(3)
    mel_t = rng.uniform(0, 1, (3, hp.max_iters * hp.outputs_per_step, hp.num_mels)).astype(np.float32)
    ref = O.tacotron_forward(small_weights, hp, ids, lengths, mel_targets=mel_t, identities=spk, id_num=6,
                             teacher_force=True, bn_mode="moving")
    eng.set_gemm_mode(mode)
    try:
        mel, lin, al, steps = eng.forward(ids, lengths, spk, mel_t, True, 0)
    finally:
        eng.set_gemm_mode(1)
    assert steps == ref["steps"]
    assert maxabs(mel, ref["mel_outputs"]) < tol and maxabs(lin, ref["linear_outputs"]) < tol


def test_tacotron_initialize_contract(small_hp, small_weights):
    """reference attribute contract (models/tacotron.py:106-113) through the host class."""
    from tacotron_multispeaker_b200.tacotron import create_model
    m = create_model("tacotron", small_hp, verbose=False)
    m.load_weights(small_weights)
    ids, lengths, spk = make_inputs(2, 15, 6, 4)
    m.initialize(ids, lengths, identities=spk, id_num=6)
    r, steps = small_hp.outputs_per_step, small_hp.max_iters
    assert tuple(m.mel_outputs.shape) == (2, steps * r, 80)
    assert tuple(m.linear_outputs.shape) == (2, steps * r, 1025)
    assert tuple(m.alignments.shape) == (2, 15, steps)
    assert m.inputs is ids and m.input_lengths is lengths and m.identities is spk
    assert m.mel_targets is None and m.linear_targets is None
    ref = O.tacotron_forward(small_weights, small_hp, ids, lengths, identities=spk, id_num=6)
    assert maxabs(m.mel_outputs, ref["mel_outputs"]) < 1e-3
    with pytest.raises(Exception):
        create_model("wavenet", small_hp)


def test_single_speaker_branch(small_hp):
    """identities None or id_num<=1 -> 256-d embedding, no speaker table (tacotron.py:48-58)."""
    from tacotron_multispeaker_b200.tacotron import Tacotron
    from tacotron_multispeaker_b200.weights import random_init
    w = random_init(small_hp, 0, seed=3, randomize_bn=True)
    m = Tacotron(small_hp, verbose=False)
    m.load_weights(w)
    ids, lengths, _ = make_inputs(2, 12, 1, 5)
    m.initialize(ids, lengths)
    ref = O.tacotron_forward(w, small_hp, ids, lengths)
    assert maxabs(m.mel_outputs, ref["mel_outputs"]) < 1e-3
    assert maxabs(m.linear_outputs, ref["linear_outputs"]) < 1e-3


def test_stop_token_kat(small_hp):
    """Zero output projection -> every sample finishes at step 0 (all outputs == 0.0):
    steps == 1 and mel_outputs is [N, r, 80] of zeros (helpers.py:35, SURVEY 8c KAT 10)."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.weights import random_init
    w = random_init(small_hp, 0, seed=9)
    w["model/inference/decoder/output_projection_wrapper/kernel"][:] = 0.0
    w["model/inference/decoder/output_projection_wrapper/bias"][:] = 0.0
    e = Engine(small_hp, 0)
    e.load_weights(w)
    ids, lengths, _ = make_inputs(3, 9, 1, 6)
    mel, lin, al, steps = e.forward(ids, lengths)
    assert steps == 1
    assert tuple(mel.shape) == (3, small_hp.outputs_per_step, 80) and float(mel.abs().max()) == 0.0
    assert tuple(lin.shape) == (3, small_hp.outputs_per_step, 1025)
    assert tuple(al.shape) == (3, 9, 1)
    ref = O.tacotron_forward(w, small_hp, ids, lengths)
    assert ref["steps"] == 1
    assert maxabs(lin, ref["linear_outputs"]) < 1e-3
    e.close()


def test_stop_token_kat_host_path(small_hp):
    """The same early stop through taco_forward_host_begin/_wait/_end: the forward is enqueued for max_iters steps
    (optimistic), _end finds steps == 1 and redoes the post-net on the true length before returning."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.weights import random_init
    hp = small_hp
    w = random_init(hp, 0, seed=9)
    w["model/inference/decoder/output_projection_wrapper/kernel"][:] = 0.0
    w["model/inference/decoder/output_projection_wrapper/bias"][:] = 0.0
    e = Engine(hp, 0)
    e.load_weights(w)
    N, T_in = 3, 9
    ids, lengths, _ = make_inputs(N, T_in, 1, 6)
    ms = e.max_steps(False, 0)
    mel = np.full((N, ms * hp.outputs_per_step, 80), 7.0, np.float32)
    lin = np.full((N, ms * hp.outputs_per_step, 1025), 7.0, np.float32)
    al = np.zeros((N, T_in, ms), np.float32)
    e.forward_host_begin(ids, lengths, None, None, False, 0, mel, lin, al)
    e.forward_host_wait(0)
    e.forward_host_wait(1)
    steps = e.forward_host_end()
    assert steps == 1
    ref = O.tacotron_forward(w, hp, ids, lengths)
    r = hp.outputs_per_step
    assert float(np.abs(mel[:, :r]).max()) == 0.0
    assert maxabs(torch.from_numpy(lin[:, :r]), ref["linear_outputs"]) < 1e-3
    e.close()


def test_forward_host_matches_device(eng, small_hp):
    hp = small_hp
    N, T_in = 3, 14
    ids, lengths, spk = make_inputs(N, T_in, 6, 21)
    mel_d, lin_d, al_d, steps = eng.forward(ids, lengths, spk)
    ms = eng.max_steps(False)
    mel = np.zeros((N, ms * hp.outputs_per_step, 80), np.float32)
    lin = np.zeros((N, ms * hp.outputs_per_step, 1025), np.float32)
    al = np.zeros((N, T_in, ms), np.float32)
    s2 = eng.forward_host(ids, lengths, spk, None, False, 0, mel, lin, al)
    assert s2 == steps
    assert np.array_equal(mel, mel_d.cpu().numpy())
    assert np.array_equal(lin, lin_d.cpu().numpy())
    assert np.array_equal(al, al_d.cpu().numpy())


def test_r1_fork_defaults():
    """The fork's own hparams (outputs_per_step=1) go through the same kernels."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=1, max_iters=12)
    w = random_init(hp, 4, seed=5, randomize_bn=True)
    e = Engine(hp, 4)
    e.load_weights(w)
    ids, lengths, spk = make_inputs(3, 10, 4, 8)
    mel, lin, al, steps = e.forward(ids, lengths, spk)
    ref = O.tacotron_forward(w, hp, ids, lengths, identities=spk, id_num=4)
    assert steps == ref["steps"] == 12
    assert maxabs(mel, ref["mel_outputs"]) < 1e-3
    assert maxabs(lin, ref["linear_outputs"]) < 1e-3
    e.close()


def test_full_size_free_running_config3():
    """BASELINE config 3 at full size (batch 32, T_in 100, 200 decoder steps x r=5 = 1000 frames, free running):
    mel / linear within the north-star 1e-3 of the oracle, alignments within 1e-5 with identical per-step argmax,
    identical stop step.  The decoder runs on the mma.sync kernel with 7 clusters of 5/4 utterances."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    w = random_init(hp, 60, seed=1234)
    ids, lengths, spk = make_inputs(32, 100, 60, 1, min_len=60, vocab=(7108, 7325))
    ref = O.tacotron_forward(w, hp, ids, lengths, identities=spk, id_num=60)
    e = Engine(hp, 60)
    e.load_weights(w)
    mel, lin, al, steps = e.forward(ids, lengths, spk)
    geo = e.decoder_geometry(32)
    e.close()
    assert steps == ref["steps"] == 200
    assert geo["cluster_size"] == 16 and geo["num_clusters"] * geo["samples_per_cluster"] >= 32
    assert maxabs(mel, ref["mel_outputs"]) < 1e-3
    assert maxabs(lin, ref["linear_outputs"]) < 1e-3
    assert maxabs(al, ref["alignments"]) < 1e-5
    assert torch.equal(al.cpu().argmax(dim=1), ref["alignments"].argmax(dim=1))


@pytest.mark.parametrize("bn_mode", ["batch", "moving"])
def test_full_size_teacher_forced_config2(bn_mode):
    """BASELINE config 2 at full size (batch 32, T_in 100, 1000 target frames -> 200 teacher-forced steps, r=5), in the reference's
    own training-graph semantics (batch-statistics BN, `is_training` keyed off linear_targets: models/tacotron.py:36) and with
    moving statistics: mel / linear within the north-star 1e-3 of the oracle, identical per-step attention argmax."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    w = random_init(hp, 60, seed=1234, randomize_bn=True)
    ids, lengths, spk = make_inputs(32, 100, 60, 2, min_len=60, vocab=(7108, 7325))
    mel_t = np.random.default_rng(22).uniform(0, 1, (32, 1000, hp.num_mels)).astype(np.float32)
    ref = O.tacotron_forward(w, hp, ids, lengths, mel_targets=mel_t, identities=spk, id_num=60, teacher_force=True, bn_mode=bn_mode)
    e = Engine(hp, 60)
    e.load_weights(w)
    mel, lin, al, steps = e.forward(ids, lengths, spk, mel_t, True, 1 if bn_mode == "batch" else 0)
    e.close()
    assert steps == ref["steps"] == 200
    assert maxabs(mel, ref["mel_outputs"]) < 1e-3
    assert maxabs(lin, ref["linear_outputs"]) < 1e-3
    assert maxabs(al, ref["alignments"]) < 1e-5
    assert torch.equal(al.cpu().argmax(dim=1), ref["alignments"].argmax(dim=1))


def test_forward_is_deterministic_under_repetition():
    """compute-sanitizer is closed on this pool, so races in the cluster decoder (st.async / mbarrier exchanges, named-barrier
    handoffs between the critical and background warps), the cp.async BiGRU and the tcgen05 pipelines are looked for the other
    way: no kernel uses atomics on its data path, so every output must be BIT-identical from run to run.  Twelve full-size
    forwards (config 3: 7 clusters x 16 CTAs, 200 steps) and twelve batch-1 forwards (critical-group attention), interleaved with
    a second handle on another stream that keeps the other SMs busy."""
    from tacotron_multispeaker_b200.engine import Engine
    from tacotron_multispeaker_b200.hparams import HParams
    from tacotron_multispeaker_b200.weights import random_init
    hp = HParams(outputs_per_step=5, max_iters=200)
    w = random_init(hp, 60, seed=1234)
    dev = torch.device("cuda", 0)
    e = Engine(hp, 60); e.load_weights(w)
    noise = Engine(hp, 60); noise.load_weights(w)
    side = torch.cuda.Stream(device=dev)
    try:
        for N, T_in in ((32, 100), (1, 77), (2, 60)):
            ids, lengths, spk = make_inputs(N, T_in, 60, 7 + N, min_len=max(1, T_in // 2), vocab=(7108, 7325))
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
                        assert torch.equal(a_, b_), "N=%d: run %d differs from run 0" % (N, rep)
    finally:
        e.close(); noise.close()


@pytest.mark.parametrize("N,S", [(1, 1), (7, 1), (13, 2), (8, 8), (23, 3), (40, 8)])
def test_decode_mma_cluster_cuts(eng, ow, small_hp, N, S):
    """The mma.sync decoder cuts a batch into clusters of S <= 8 utterances (uneven cuts, more clusters than fit at
    once -> several waves): every cut gives the oracle's result."""
    e_dec, e_al, al, ral = _decode_case(eng, ow, small_hp, N, 37, True, 100 + N, S)
    assert e_dec < 2e-4 and e_al < 1e-5
    assert torch.equal(al.cpu().argmax(dim=1), ral.argmax(dim=1))
    e_dec, e_al, _, _ = _decode_case(eng, ow, small_hp, N, 37, False, 200 + N, S)
    assert e_dec < 1e-3 and e_al < 1e-4


def test_forward_host_validates_buffers(eng, small_hp):
    """The host entry points take raw pointers: default-dtype (int64 / float64) inputs are converted, output buffers of the
    wrong dtype, layout or size are refused instead of being reinterpreted or overrun."""
    hp = small_hp
    ids, lengths, spk = make_inputs(2, 9, 6, 5)
    ms = eng.max_steps(False)
    T = ms * hp.outputs_per_step
    mel = np.zeros((2, T, hp.num_mels), np.float32); lin = np.zeros((2, T, hp.num_freq), np.float32)
    al = np.zeros((2, 9, ms), np.float32)
    s_ref = eng.forward_host(ids, lengths, spk, None, False, 0, mel, lin, al)
    mel64 = np.zeros_like(mel)
    s2 = eng.forward_host(ids.astype(np.int64), lengths.astype(np.int64), spk.astype(np.int64), None, False, 0, mel64, None, None)
    assert s2 == s_ref and np.array_equal(mel64, mel)
    with pytest.raises(TypeError):
        eng.forward_host(ids, lengths, spk, None, False, 0, mel.astype(np.float64), lin, al)
    with pytest.raises(TypeError):
        eng.forward_host(ids, lengths, spk, None, False, 0, mel, lin.transpose(0, 2, 1).copy().transpose(0, 2, 1), al)
    with pytest.raises(ValueError):
        eng.forward_host(ids, lengths, spk, None, False, 0, mel[:, : T - 1].copy(), lin, al)
    with pytest.raises(ValueError):
        eng.forward_host(ids, lengths[:1], spk, None, False, 0, mel, lin, al)


def test_forward_cuda_graph_replay(small_weights, small_hp):
    """The same forward call (same device pointers, shapes, modes) on a non-default stream is captured into a CUDA graph on
    its second arrival and replayed afterwards: results must be bit-identical to plain launches, the launch counter keeps
    counting the kernels inside the graph, and a call with other pointers falls back to plain launches."""
    hp = small_hp
    ids, lengths, spk = make_inputs(3, 19, 6, 21)
    from tacotron_multispeaker_b200.engine import Engine
    dev = torch.device("cuda", 0)
    e_plain = Engine(hp, 6); e_plain.load_weights(small_weights); e_plain.set_cuda_graphs(False)
    e_graph = Engine(hp, 6); e_graph.load_weights(small_weights)
    try:
        ref = e_plain.forward(ids, lengths, spk)
        ids_d, len_d, spk_d = (torch.from_numpy(x).to(dev) for x in (ids, lengths, spk))
        ms = e_graph.max_steps(False)
        T = ms * hp.outputs_per_step
        out = (torch.zeros(3, T, hp.num_mels, device=dev), torch.zeros(3, T, hp.num_freq, device=dev), torch.zeros(3, 19, ms, device=dev))
        st = torch.cuda.Stream(device=dev)
        st.wait_stream(torch.cuda.current_stream())
        counts = []
        with torch.cuda.stream(st):
            for rep in range(4):        # plain, capture + launch, replay, replay
                for o in out:
                    o.zero_()
                c0 = e_graph.launch_count()
                mel, lin, al, s = e_graph.forward(ids_d, len_d, spk_d, out=out)
                st.synchronize()
                counts.append(e_graph.launch_count() - c0)
                assert s == ref[3]
                for got, want in zip((mel, lin, al), ref[:3]):
                    assert torch.equal(got, want), "rep %d differs from plain launches" % rep
            # other pointers: plain launches again, still correct
            mel2, lin2, al2, s2 = e_graph.forward(ids, lengths, spk)
            st.synchronize()
            assert torch.equal(lin2, ref[1])
        assert len(set(counts)) == 1 and counts[0] > 25, counts
    finally:
        e_plain.close(); e_graph.close()


def test_forward_host_begin_end(eng, small_hp):
    """taco_forward_host == taco_forward_host_begin + taco_forward_host_end (outputs land after _end)."""
    hp = small_hp
    N, T_in = 3, 14
    ids, lengths, spk = make_inputs(N, T_in, 6, 21)
    ms = eng.max_steps(False)
    shapes = ((N, ms * hp.outputs_per_step, 80), (N, ms * hp.outputs_per_step, 1025), (N, T_in, ms))
    a = [np.zeros(s, np.float32) for s in shapes]
    b = [np.zeros(s, np.float32) for s in shapes]
    s1 = eng.forward_host(ids, lengths, spk, None, False, 0, *a)
    eng.forward_host_begin(ids, lengths, spk, None, False, 0, *b)
    s2 = eng.forward_host_end()
    assert s1 == s2
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
