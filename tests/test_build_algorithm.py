"""The device construction ALGORITHM (tests/build_algorithm.py models build_kernels.cu step by step) against the oracle's
literal restatement of BVHAccelerator::construct: key reductions reproduce the ordered fold down to the sign of a zero, the
closed-form permutation reproduces libstdc++'s Hoare partition, chain lengths reproduce the pre-order numbering.  Runs without
a GPU; where the reference libraries exist it also throws random tie-heavy inputs at the reference itself."""
import numpy as np
import pytest

import build_algorithm
import bvhcases

SMALL = {k: v for k, v in bvhcases.cases(big=1500).items() if len(v[0]) <= 1500}


@pytest.mark.parametrize("name", sorted(SMALL))
def test_device_algorithm_equals_the_oracle(oracle_port, name):
    bounds, non_tri, first_id = SMALL[name]
    want = oracle_port.build_bvh(bounds, non_tri, first_id)
    nodes, order, n_internal, depth = build_algorithm.build(bounds, non_tri, first_id)
    assert n_internal == want["head"]["n_nodes"] and depth == want["head"]["max_depth"]
    assert np.array_equal(order, want["order"])
    assert nodes.tobytes() == want["nodes"].tobytes()


def test_tie_heavy_inputs_against_the_live_reference(oracle_port):
    """Coordinates drawn from a handful of values (signed zeros among them): ties in every fold and every partition."""
    from oracle import ref
    if not ref.available():
        pytest.skip("reference library not built (needs the reference sources: SP_REFERENCE, or a checkout named reference beside the repository)")
    rng = np.random.default_rng(99)
    values = np.array([-0.0, 0.0, -1.0, 1.0, 0.5, 2.0, -2.0], dtype=np.float32)
    for trial in range(200):
        n = int(rng.integers(0, 40))
        a, b = values[rng.integers(0, len(values), (n, 3))], values[rng.integers(0, len(values), (n, 3))]
        lo = np.where(a < b, a, np.where(b < a, b, a))      # keep the signs of zeros as drawn
        hi = np.where(a < b, b, np.where(b < a, a, b))
        bounds = np.concatenate([lo, hi], axis=1).astype(np.float32)
        want = ref.build_bvh(bounds, None, 0)
        got = oracle_port.build_bvh(bounds, None, 0)
        assert not bvhcases.same(got, want), (trial, bvhcases.same(got, want))
        assert got["root_bounds"].tobytes() == want["root_bounds"].tobytes()
        nodes, order, n_internal, depth = build_algorithm.build(bounds, None, 0)
        assert n_internal == want["head"]["n_nodes"] and depth == want["head"]["max_depth"], trial
        assert np.array_equal(order, want["order"]) and nodes.tobytes() == want["nodes"].tobytes(), trial
