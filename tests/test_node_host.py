"""The bound node's host logic on CPU: a gossip simulation (real Ed25519 signatures, BLAKE2b ids, random peers)
runs over `bind(host)` with the oracle standing in for the device, over the tests' own host; every node's state must
equal a replay of its own arrival trace and call schedule through the oracle.  Node traces recorded from this
simulation and from the reference's own driver over `bind(swirld.Node)` are replayed against the unmodified
reference's results on them (tests/golden)."""
import numpy as np
import pytest

import golden_specs as gs
import node_sim
from oracle_engine import OracleEngine
from swirld_b200.traces import Trace
from util import assert_same, load_golden

KEYS = ["round", "famous", "consensus", "transactions"]


@pytest.fixture(scope="module")
def sim():
    return node_sim.run_sim(4, 400, OracleEngine, capacity=64, seed=5)   # small capacity: forces growth replay


def test_transactions_are_consistent(sim):
    # prefix agreement between nodes is NOT a property of the reference (its final order
    # depends on each node's call schedule, SURVEY.md section 0.5); each node's own state is
    # pinned against the oracle / the reference below.
    for nd in sim:
        assert len(nd.transactions) > 20
        assert len(set(nd.transactions)) == len(nd.transactions)


def test_views_and_attributes(sim):
    nd = sim[0]
    h = nd.head
    assert nd.hg[h].c == nd.pk and nd.height[h] >= 1
    assert nd.can_see[h][nd.pk] == h
    assert nd.round[h] >= nd.round[nd.hg[h].p[0]]
    assert set(nd.idx) == set(nd.transactions)
    assert [nd.idx[x] for x in nd.transactions] == list(range(len(nd.transactions)))
    assert nd.tbd == set(nd.hg) - set(nd.transactions)
    r0 = nd.witnesses[0]
    assert set(r0) <= set(nd.stake) and all(nd.round[w] == 0 for w in r0.values())
    fam = [x for x in nd.hg if x in nd.famous]
    assert fam and all(isinstance(nd.famous[x], bool) for x in fam)
    assert nd.famous.get(b"nope") is None
    with pytest.raises(KeyError):
        nd.round[b"nope"]


def test_each_node_matches_oracle_replay(sim):
    for nd in sim:
        tr, sizes = node_sim.node_trace(nd)
        assert_same(node_sim.replay_oracle(tr, sizes), node_sim.node_results(nd), KEYS, "node vs oracle replay")


def test_each_node_matches_reference_replay():
    """Node traces and call schedules recorded from one run of this simulation, with the reference's replay of each
    (gs.NODE_SIM, recorded by oracle/make_golden.py): the oracle's replay must reproduce it.  Every live node is tied
    to the oracle's replay by test_each_node_matches_oracle_replay."""
    for name in gs.NODE_SIM:
        g = load_golden(name)
        tr = Trace(int(g["M"]), g["p0"], g["p1"], g["creator"], g["t"], g["sig"], name)
        assert_same(g, node_sim.replay_oracle(tr, g["sizes"].tolist()), KEYS, name + ": oracle replay vs reference replay")


def test_drop_in_for_the_reference_drivers():
    """`swirld.Node = bind(swirld.Node)` before `swirld.test(4, 300)`: what the reference's own driver, main loop and
    sync fed every node (its arrival trace and call schedule, gs.DROP_IN, recorded by oracle/make_golden.py) is fed
    again to a bound node; its state must equal the reference's replay of the same trace and schedule."""
    for name in gs.DROP_IN:
        g = load_golden(name)
        nd = node_sim.replay_node(g, OracleEngine)
        tr, sizes = node_sim.node_trace(nd)
        assert sizes == g["sizes"].tolist()
        assert all(np.array_equal(getattr(tr, k), g[k]) for k in ("p0", "p1", "creator", "t", "sig"))
        assert len(nd.transactions) > 5
        assert_same(g, node_sim.node_results(nd), KEYS, name + ": drop-in node vs reference")


def test_forked_events_are_dropped_not_fatal():
    """A Byzantine peer's fork (a second event on the same self-parent) is treated as invalid: the node keeps working
    and its device state stays consistent (the reference would accept the fork; the engine's contract is fork-free)."""
    import host_sim
    nodes = node_sim.run_sim(3, 60, OracleEngine, seed=9)
    a, b = nodes[0], nodes[1]
    # b forges a sibling of its own head: same self-parent, other other-parent
    sp = b.hg[b.head].p
    assert sp
    other = next(h for h in b.hg if b.hg[h].c != b.pk and h != sp[1])
    h2, ev2 = host_sim.HostNode.new_event(b, "fork", (sp[0], other))
    assert host_sim.HostNode.is_valid_event(a, h2, ev2) or other not in a.hg or sp[0] not in a.hg
    n_before = len(a.hg)
    if sp[0] in a.hg and other in a.hg and a._heads.get(b.pk) != sp[0]:
        assert not a.is_valid_event(h2, ev2)             # a already holds b's real event on that self-parent
    # a second root is always a fork
    hr, evr = host_sim.HostNode.new_event(b, None, ())
    assert not a.is_valid_event(hr, evr)
    assert len(a.hg) == n_before
    loop = a.main()
    next(loop)
    loop.send(None)                                      # the node still gossips and advances
    assert len(a.hg) > n_before
    tr, sizes = node_sim.node_trace(a)
    assert_same(node_sim.replay_oracle(tr, sizes), node_sim.node_results(a), KEYS, "after the rejected fork")


def test_non_integral_stake_is_refused():
    import host_sim
    import sodium
    kp = sodium.crypto_sign_keypair()
    with pytest.raises(ValueError):
        node_sim.bound_class(host_sim.HostNode, OracleEngine)(kp, {}, 1, {kp[0]: 1.5})
