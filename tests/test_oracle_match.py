"""CPU tests: the matchToMap oracle (oracle/match_oracle.c) against (a) golden vectors dumped from the reference's own Mapper
(tools/make_golden_match.py) and (b) the reference, live or recorded.  Exact: identical keypoint -> map point maps."""
import numpy as np
import pytest

from conftest import golden
from alvaar_b200 import synth
from match_util import oracle_match, reference_match


def problem(seed):
    return synth.make_match_problem(seed, n_frame_kp=150 + 20 * seed, n_local=350 + 50 * seed)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
@pytest.mark.parametrize("nkp3d", [100, 10])
def test_match_golden(oracle, seed, nkp3d):
    import hashlib
    g = golden("match")
    p = problem(seed)
    h = hashlib.sha256()
    for k in sorted(p):
        if isinstance(p[k], np.ndarray):
            h.update(np.ascontiguousarray(p[k]).tobytes())
    assert h.hexdigest() == str(g[f"s{seed}_sha"]), "synthetic map generator changed: re-dump the golden"
    m = oracle_match(oracle, p, g[f"s{seed}_{nkp3d}_order"], nkp3d)
    assert len(m) > 40
    assert sorted(m) == g[f"s{seed}_{nkp3d}_kp"].tolist()
    assert [m[k] for k in sorted(m)] == g[f"s{seed}_{nkp3d}_mp"].tolist()


@pytest.mark.parametrize("seed", [11, 12, 13, 14, 15, 16])
def test_match_live_reference(oracle, ref_results, seed):
    p = synth.make_match_problem(seed, n_frame_kp=120 + 13 * (seed % 5), n_local=300 + 37 * (seed % 7), dup_frac=0.5)
    for nk in (100, 5):
        def match():
            order, m = reference_match(ref_results.lib, p, nk)
            return (order, np.array(sorted(m.items()), np.int32).reshape(-1, 2))
        order, want = ref_results.get(f"match/{seed}/{nk}", match)
        want = dict(want.tolist())
        assert oracle_match(oracle, p, order, nk) == want and len(want) > 30


def test_match_order_decides_ties(oracle):
    """Two local map points that are exact copies of each other (same world point, same descriptors, disjoint keyframes from the
    keypoint): the one processed LAST wins the keypoint (mapper.cpp:565-585, `<=`)."""
    p = synth.make_match_problem(3)
    order = p["local_ids"]
    m1 = oracle_match(oracle, p, order, 100)
    m2 = oracle_match(oracle, p, order[::-1].copy(), 100)
    assert set(m1) == set(m2)          # the same keypoints get matched ...
    assert len(m1) > 40                # ... (possibly to a different duplicate when two tie)
