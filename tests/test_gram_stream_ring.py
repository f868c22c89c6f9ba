"""The bf16x2 Gram kernel (64 <= N_pad <= 112 clients, D >= 32768) with many k-blocks per CTA.

The kernel streams one 64-column k-block per step through a 7-slot shared-memory ring that four converter warps and
two MMA issuers rotate over.  The other GPU tests give each CTA only a few k-blocks; here D = 32,785 gives fewer
k-blocks per CTA than slots, and D = 1,000,003 gives about a hundred, so the ring wraps many times and the
accumulation chains end on odd tails.  Both have a ragged last k-block.  The client counts cover every N_pad class
(64, 80, 96, 112); n = 49, 90, 97 and 100 leave the last real 8-row unit partly filled.
"""
import numpy as np
import pytest

from oracle import c_oracle as co, ref_numpy as orc

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N_VALUES = [49, 64, 80, 90, 96, 97, 100, 112]     # N_pad 64, 64, 80, 96, 96, 112, 112, 112
D_SHORT, D_LONG = 32768 + 17, 1_000_003


def hetero(rng, n, d):
    return (0.1 * rng.standard_normal(d) + np.exp(0.25 * rng.standard_normal((n, 1))) * rng.standard_normal((n, d))).astype(np.float32)


def padded(G):
    """Device copy with a pitch that is a multiple of 4 floats (16 bytes), as the TMA path needs."""
    n, d = G.shape
    Gp = torch.zeros((n, (d + 3) // 4 * 4), device="cuda")[:, :d]
    Gp.copy_(torch.from_numpy(G))
    return Gp


@pytest.fixture(scope="module")
def api():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    from attacking_federate_learning_b200 import _device, _native
    _native.lib()
    return _device, _native


@pytest.mark.parametrize("d", [D_SHORT, D_LONG])
@pytest.mark.parametrize("n", N_VALUES)
def test_ring_matches_oracle(api, n, d):
    dev, nat = api
    rng = np.random.default_rng(n * 7 + (d & 0xFF))
    G = hetero(rng, n, d)
    Gp = padded(G)
    flags = nat.GRAM_FORCE_TCGEN05 | nat.GRAM_BF16X2
    d2 = dev.sqdist_partial(Gp, flags).cpu().numpy()
    ref = co.pairwise_sqdist(G)
    off = ~np.eye(n, dtype=bool)
    rel = (d2[off] - ref[off]) / ref[off]
    # same caps as test_krum_matches_oracle: a uniform bias from the dropped b2*b2 term, a small pair-to-pair spread
    assert np.abs(rel).max() < 8e-6, np.abs(rel).max()
    assert rel.max() - rel.min() < 3e-6, (rel.min(), rel.max())
    assert np.array_equal(d2, d2.T) and not d2.diagonal().any()
    again = dev.sqdist_partial(Gp, flags).cpu().numpy()
    assert np.array_equal(d2.view(np.uint64), again.view(np.uint64))


def test_identical_rows_across_units(api):
    """Rows 0..f-1 (across the 8-row unit edge at 7/8) and rows 95/99 (the last, partly filled unit) are copies."""
    dev, nat = api
    n, d, f = 100, D_LONG, 24
    rng = np.random.default_rng(11)
    G = 5.0 * hetero(rng, n, d)
    G[:f] = 0.002 * G[f]
    G[99] = G[95]
    Gp = padded(G)
    for flags in (nat.GRAM_FORCE_TCGEN05 | nat.GRAM_BF16X2, 0):
        d2 = dev.sqdist_partial(Gp, flags)
        assert float(d2[:f, :f].abs().max()) == 0.0
        assert float(d2[95, 99]) == 0.0 and float(d2[99, 95]) == 0.0
        dist = dev.sqdist_to_dist(d2)
        assert all(torch.equal(dist[0, f:], dist[i, f:]) for i in range(1, f))
        assert torch.equal(dist[95, :95], dist[99, :95])
        assert int(dev.krum_select(dist, n, f).item()) == 1
    assert orc.krum_select(np.sqrt(co.pairwise_sqdist(G)), orc.visit_order(n), n, f, dtype=np.float64) == 1


def test_fused_krum_step_long_stream(api):
    """ShardedAggregator().krum runs the Gram kernel, the reduction, the d2 table and the Krum tail as one step."""
    from attacking_federate_learning_b200.sharded import ShardedAggregator
    n, d, f = 100, 1_000_004, 24
    rng = np.random.default_rng(3)
    G = hetero(rng, n, d)
    table64 = np.sqrt(co.pairwise_sqdist(G))
    want, margin = orc.krum_select(table64, orc.visit_order(n), n, f, dtype=np.float64, with_margin=True)
    assert margin > 1e-5, "test input has a near-tie; pick another seed"
    Gd = torch.from_numpy(G).cuda()
    assert ShardedAggregator().krum(Gd, n, f, return_index=True) == want
