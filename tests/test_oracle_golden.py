"""Pin oracle/ref_numpy.py to outputs of the unmodified reference — bit for bit: the edge cases and
shapes of tests/golden/golden_v1.npz (tests/golden/make_golden.py) and the seeded random cases of
tests/golden/golden_seeded_v1.npz (tests/golden/make_golden_seeded.py)."""
import os

import numpy as np
import pytest

from conftest import ROOT, golden_names
from oracle import ref_numpy as orc


def same_bits(a, b):
    a = np.asarray(a); b = np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("name", golden_names("dist"))
def test_distances_and_order(golden, name):
    G = golden[f"{name}/G"]
    assert same_bits(orc.pairwise_distances_f32(G), golden[f"{name}/dist"])
    assert orc.visit_order(len(G)) == list(golden[f"{name}/order"])
    # the float64 arbiter agrees with the fp32 table to fp32 rounding noise
    np.testing.assert_allclose(orc.pairwise_distances_f64(G), golden[f"{name}/dist"], rtol=2e-6, atol=1e-7)


@pytest.mark.parametrize("name", golden_names("krum_idx"))
def test_krum_index(golden, name):
    G = golden[f"{name}/G"]; f = int(golden[f"{name}/f"])
    assert orc.krum(G, len(G), f, return_index=True) == int(golden[f"{name}/krum_idx"])


def test_krum_returns_view(golden):
    G = golden["het_n10_d64_f2/G"].copy()
    row = orc.krum(G, 10, 2)
    assert row.base is G or np.shares_memory(row, G)


@pytest.mark.parametrize("name", golden_names("tm"))
def test_trimmed_mean(golden, name):
    G = golden[f"{name}/G"]; f = int(golden[f"{name}/f"])
    assert same_bits(orc.trimmed_mean(G, len(G), f), golden[f"{name}/tm"])
    np.testing.assert_allclose(orc.trimmed_mean_f64(G, len(G), f), golden[f"{name}/tm"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("name", golden_names("bulyan"))
def test_bulyan(golden, name):
    G = golden[f"{name}/G"]; f = int(golden[f"{name}/f"]); n = len(G)
    table = orc.pairwise_distances_f32(G)
    assert orc.bulyan_select(table, n, f) == list(golden[f"{name}/bulyan_sel"])
    assert same_bits(orc.bulyan(G, n, f), golden[f"{name}/bulyan"])


@pytest.mark.parametrize("name", golden_names("mean"))
def test_mean(golden, name):
    G = golden[f"{name}/G"]
    assert same_bits(orc.no_defense(G), golden[f"{name}/mean"])


@pytest.mark.parametrize("nm", ["a", "b", "c", "d"])
def test_alie(golden, nm):
    rows = golden[f"alie_{nm}/rows"]; z = float(golden[f"alie_{nm}/z"])
    crafted, mu, sigma = orc.alie_attack([r.copy() for r in rows], z)
    assert same_bits(mu, golden[f"alie_{nm}/mean"])
    assert same_bits(sigma, golden[f"alie_{nm}/stdev"])
    if z == 0:
        assert crafted is None and same_bits(golden[f"alie_{nm}/grads0"], rows[0])
    else:
        assert crafted is mu and same_bits(crafted, golden[f"alie_{nm}/grads0"])
        assert bool(golden[f"alie_{nm}/aliased"])


def _fake_training(p):                                   # the stand-in make_golden_backdoor.py used for backdoor.py:108
    return (p * np.float32(0.9) + np.float32(0.01)).astype(np.float32)


@pytest.mark.parametrize("nm", ["d8", "d1000", "d4099_tight", "d257_wide"])
def test_backdoor_hook(golden_backdoor, nm):
    g = golden_backdoor
    got = orc.backdoor_attack_grads(g[f"hook_{nm}/mean"].copy(), g[f"hook_{nm}/stdev"].copy(), g[f"hook_{nm}/params"].copy(),
                                    float(g[f"hook_{nm}/lr"]), float(g[f"hook_{nm}/z"]), _fake_training)
    assert same_bits(got, g[f"hook_{nm}/want"])


@pytest.mark.parametrize("nm", ["f5_d300", "f24_d2051"])
def test_backdoor_attack(golden_backdoor, nm):
    g = golden_backdoor
    mu, sigma = orc.alie_stats([r.copy() for r in g[f"attack_{nm}/rows"]])
    assert same_bits(mu, g[f"attack_{nm}/mean"]) and same_bits(sigma, g[f"attack_{nm}/stdev"])
    got = orc.backdoor_attack_grads(mu, sigma, g[f"attack_{nm}/params"], float(g[f"attack_{nm}/lr"]),
                                    float(g[f"attack_{nm}/z"]), _fake_training)
    assert same_bits(got, g[f"attack_{nm}/grads0"]) and bool(g[f"attack_{nm}/aliased"])


def test_edge_semantics(golden):
    # SURVEY section 4 table
    assert int(golden["tie012_win/krum_idx"]) == 1                      # ties -> user 1 beats user 0
    assert float(golden["tm_tie_a/tm"][0]) == -0.5 and float(golden["tm_tie_b/tm"][0]) == 0.5
    assert int(golden["n1/krum_idx"]) == -1
    with pytest.raises(AssertionError):
        orc.krum(golden["het_n10_d64_f2/G"], 10, 5)                     # n >= 2f+1
    with pytest.raises(AssertionError):
        orc.bulyan(golden["het_n10_d64_f2/G"], 10, 2)                   # n >= 4f+3
    # NaN inputs: Python's sorted() on a list holding NaN is order-dependent, so the reference's
    # answer is not a function of the values alone -> documented as undefined, not pinned.


@pytest.fixture(scope="module")
def golden_seeded():
    return np.load(os.path.join(ROOT, "tests", "golden", "golden_seeded_v1.npz"), allow_pickle=False)


@pytest.mark.parametrize("seed", range(6))
def test_against_live_reference(golden_seeded, seed):
    """Random N, D, f (identical leading rows for odd seeds): every rule and the ALIE attack against what the
    reference returned on the same matrix."""
    g = {k.split("/", 1)[1]: golden_seeded[k] for k in golden_seeded.files if k.startswith(f"seed{seed}/")}
    G, f = g["G"], int(g["f"]); n = len(G)
    assert orc.krum(G, n, f, return_index=True) == int(g["krum_idx"])
    assert same_bits(orc.trimmed_mean(G, n, f), g["tm"])
    assert same_bits(orc.no_defense(G), g["mean"])
    if n >= 4 * f + 3:
        assert same_bits(orc.bulyan(G, n, f), g["bulyan"])
    crafted, mu, sigma = orc.alie_attack([G[i].copy() for i in range(max(f, 1))], float(g["alie_z"]))
    assert same_bits(crafted, g["alie_grads0"]) and same_bits(sigma, g["alie_stdev"])
