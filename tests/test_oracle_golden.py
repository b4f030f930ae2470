"""Pins the oracle (oracle/swirld_oracle.c) to the reference: every committed
fixture under tests/golden/ was produced by the UNMODIFIED reference
(oracle/make_golden.py); the C restatement must reproduce it bit for bit --
rounds, witness table, famous tri-state, consensus set, per-call new_c and the
final consensus order -- under the same call schedule."""
import hashlib

import numpy as np
import pytest

import golden_specs as gs
import oracle as orc
from util import assert_same, load_golden

SMALL = [n for n in gs.SPECS if gs.SPECS[n][1]["N"] <= 20000]
LARGE = [n for n in gs.SPECS if gs.SPECS[n][1]["N"] > 20000]


def _check(name):
    tr, K, stake = gs.make_trace(name)
    g = load_golden(name)
    sha = hashlib.sha256(tr.p0.tobytes() + tr.p1.tobytes() + tr.creator.tobytes() + tr.t.tobytes()
                         + tr.sig.tobytes()).digest()
    assert bytes(g["trace_sha256"]) == sha, "trace generator drifted from the fixture"
    o = orc.run_oracle(tr, K, stake)
    assert_same(g, o, what=name)
    cs = o["oracle"].can_see()
    assert bytes(g["can_see_sha256"]) == hashlib.sha256(cs.tobytes()).digest(), name + ": can_see differs"
    if "can_see" in g:
        assert np.array_equal(g["can_see"], cs)


@pytest.mark.parametrize("name", SMALL)
def test_oracle_matches_reference_fixture(name):
    _check(name)


@pytest.mark.parametrize("name", LARGE)
def test_oracle_matches_reference_fixture_large(name):
    _check(name)


@pytest.mark.parametrize("M,N,K,seed", gs.SPOT_CASES)
def test_oracle_matches_live_reference(M, N, K, seed):
    """A gossip and an adversarial trace per case against what the reference computed on them (the fixtures
    gs.spot_names(...), recorded by oracle/make_golden.py), the whole can_see matrix included."""
    for name in gs.spot_names(M, N, K, seed):
        _check(name)
        assert "can_see" in load_golden(name)


def test_oracle_index_error_single_seer():
    """swirld.py:305 raises IndexError when only one famous witness sees an
    event; the oracle reports it instead of inventing a timestamp."""
    from swirld_b200 import traces
    tr = traces.gossip(3, 400, 3)
    try:
        orc.run_oracle(tr, 50, stake=[5, 1, 1])
    except IndexError:
        return
    # not every trace reaches that state; it must at least run clean
