"""The numpy sum-tree restatement vs the reference's golden vectors (CPU)."""
import os

import numpy as np
import pytest

from oracle.gen_golden import crc, tree_large_script, tree_script
from oracle.sumtree import SumTreeOracle


@pytest.mark.parametrize("tag,cap", [("p2", 1024), ("np2", 1000), ("tiny", 3)])
def test_tree_matches_reference_golden(golden_dir, tag, cap):
    g = np.load(os.path.join(golden_dir, "tree_small.npz"))
    tree = SumTreeOracle(cap, 0.9, 0.6)
    assert tree.num_layers == int(g[f"{tag}_num_layers"])
    for k, op in enumerate(tree_script(cap, 5)):
        if op[0] == "update":
            tree.update(op[1], op[2])
            # bit-exact: same float32 pow (numpy), same float64 child sums
            np.testing.assert_array_equal(tree.ptree, g[f"{tag}_op{k}_tree"])
        else:
            r = np.random.RandomState(op[2]).random_sample(op[1])
            idx, w = tree.sample(op[1], r)
            np.testing.assert_array_equal(idx, g[f"{tag}_op{k}_idx"])
            np.testing.assert_array_equal(w, g[f"{tag}_op{k}_isw"])


def test_tree_matches_reference_golden_large(golden_dir):
    """50,000 and 2^16 leaves: sampled indices, IS weights and the whole tree (CRC) after each round, bit-exact."""
    g = np.load(os.path.join(golden_dir, "tree_large.npz"))
    for cap, td, rounds in tree_large_script():
        tree = SumTreeOracle(cap, 0.9, 0.6)
        tree.update(np.arange(cap), td)
        for n, t2 in rounds:
            tag = f"c{cap}_n{n}"
            idx, w = tree.sample(n, np.random.RandomState(n).random_sample(n))
            np.testing.assert_array_equal(idx, g[f"{tag}_idx"])
            np.testing.assert_array_equal(w, g[f"{tag}_isw"])
            tree.update(idx, t2)
            np.testing.assert_array_equal(tree.ptree[g[f"{tag}_tree_pos"]], g[f"{tag}_tree_sample"])
            assert crc(tree.ptree) == int(g[f"{tag}_tree_crc"])
