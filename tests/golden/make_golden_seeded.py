"""Generates tests/golden/golden_seeded_v1.npz from the UNMODIFIED reference:

    python tests/golden/make_golden_seeded.py <directory of the reference checkout>

Six seeded random cases (random N, D and f, half of them with identical leading rows) fed to the reference's
defences.py (krum, trimmed_mean, no_defense, bulyan) and malicious.DriftAttack.  Each case stores its input matrix
and what the reference returned, so that tests/test_oracle_golden.py compares oracle/ref_numpy.py with the reference
bit for bit without needing the reference itself.
"""
import os
import sys

import numpy as np


class _User:                                                  # duck-typed user, as malicious.py expects
    def __init__(self, g):
        self.grads = g
        self.original_params = None
        self.learning_rate = None


def case_input(seed):
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(3, 40)); d = int(rng.integers(1, 300)); f = int(rng.integers(0, max(1, (n - 3) // 4 + 1)))
    G = (0.1 * rng.standard_normal(d) + np.exp(0.25 * rng.standard_normal((n, 1))) * rng.standard_normal((n, d))).astype(np.float32)
    if seed % 2:
        G[:max(f, 2)] = G[0]                                  # identical rows
    return G, f


def main(ref_dir):
    sys.path.insert(0, ref_dir)
    import defences as ref_def
    import malicious as ref_mal
    out = {}
    for seed in range(6):
        G, f = case_input(seed)
        n = len(G)
        k = f"seed{seed}"
        out[f"{k}/G"], out[f"{k}/f"] = G, np.int64(f)
        out[f"{k}/krum_idx"] = np.int64(ref_def.krum(G, n, f, return_index=True))
        out[f"{k}/tm"] = ref_def.trimmed_mean(G, n, f)
        out[f"{k}/mean"] = ref_def.no_defense(G, n, f)
        if n >= 4 * f + 3:
            out[f"{k}/bulyan"] = ref_def.bulyan(G, n, f)
        users = [_User(G[i].copy()) for i in range(max(f, 1))]
        att = ref_mal.DriftAttack(1.5)
        att.attack(users)
        out[f"{k}/alie_z"] = np.float64(1.5)
        out[f"{k}/alie_grads0"], out[f"{k}/alie_stdev"] = users[0].grads, att.grads_stdev
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_seeded_v1.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
