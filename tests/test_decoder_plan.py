"""Host-side decisions of the default decoder (taco_decoder_plan): where the attention operands of a cluster live for S
utterances per cluster and T_in input positions, and how many clusters a batch is cut into.  No device needed.

att_res: 3 = exp(2 key) rows and memory columns in shared memory, 4 = both in tensor memory (layout TL_ATT), 1 = keys only,
0 = neither (re-read from global memory every step)."""
import pytest

from tacotron_multispeaker_b200 import _abi

SMEM_LIMIT = 227 * 1024
BOUND = 105   # largest T_in with the attention operands on chip at S = 8

# T_in -> att_res for S = 1..8
RES = {
    1: [3, 3, 3, 3, 3, 3, 3, 3],
    37: [3, 3, 3, 3, 3, 3, 3, 4],
    60: [3, 3, 3, 3, 3, 3, 4, 4],
    100: [3, 3, 3, 3, 3, 4, 4, 4],
    BOUND: [3, 3, 3, 3, 3, 4, 4, 4],
    BOUND + 1: [3, 3, 3, 3, 4, 4, 4, 0],
    200: [3, 3, 3, 1, 1, 0, 0, 0],
    512: [3, 1, 0, 0, 0, 0, 0, 0],
}


def _plan(S, T_in):
    return _abi.decoder_plan(S, T_in, 1)   # one co-resident cluster: a batch of S is one cluster of S


@pytest.mark.parametrize("T_in", sorted(RES))
def test_attention_residency(T_in):
    got = [_plan(S, T_in) for S in range(1, 9)]
    assert [p["att_res"] for p in got] == RES[T_in]
    for S, p in zip(range(1, 9), got):
        assert p["valid"] == 1 and p["clusters"] == 1 and p["s_max"] == S
        assert p["ring_kb"] in (4, 5, 6)
        assert 0 < p["smem_bytes"] <= SMEM_LIMIT


def test_config3_resident_at_eight_per_cluster():
    """Config 3 (T_in 100): S = 8 keeps keys and memory on chip with the deepest ring; S <= 5 keeps the shared-memory plan."""
    p = _plan(8, 100)
    assert (p["att_res"], p["ring_kb"], p["smem_bytes"]) == (4, 6, 231296)
    p = _plan(5, 100)
    assert (p["att_res"], p["ring_kb"], p["smem_bytes"]) == (3, 4, 228608)


def test_bound_is_tight():
    assert all(_plan(8, T)["att_res"] == 4 for T in range(38, BOUND + 1))
    assert all(_plan(8, T)["att_res"] == 0 for T in range(BOUND + 1, 513))


@pytest.mark.parametrize("N,clusters,S", [
    (1, 1, 1),      # batch-1 latency: one cluster, critical-group attention
    (2, 1, 2),      # one cluster of 2 decodes 8 % slower than two of 1, on half the SMs
    (32, 4, 8),     # config 3: 4 clusters of 8 (64 SMs) instead of 7 of 5 (112 SMs), 18 % slower per step
    (70, 9, 8),     # two waves either way: 9 clusters of 8 instead of 14 of 5
    (256, 32, 8),   # config 4: five waves of up to 7 clusters of 8
])
def test_cluster_picker(N, clusters, S):
    for T_in in (37, 100):
        p = _abi.decoder_plan(N, T_in, 7)
        assert (p["clusters"], p["s_max"]) == (clusters, S)
        assert p["att_res"] in (3, 4)


def test_refusals():
    for N, T_in, mc in ((0, 10, 7), (4, 0, 7), (4, 513, 7), (4, 10, 0)):
        assert _abi.decoder_plan(N, T_in, mc)["valid"] == 0
