"""Helpers shared by the bound-node tests: run a gossip simulation, then replay each node's own arrival trace +
call schedule through a checker."""
import numpy as np

import host_sim
from swirld_b200 import node as gnode
from swirld_b200.traces import Trace


def bound_class(host_cls, engine_cls=None):
    """bind(host_cls); the CPU tests inject the oracle as the engine by subclassing (the product never does)."""
    cls = gnode.bind(host_cls)
    if engine_cls is None:
        return cls
    return type("GpuNodeOverOracle", (cls,), {"_engine_cls": engine_cls})


def run_sim(n_nodes, n_turns, engine_cls=None, host_cls=host_sim.HostNode, **kw):
    return host_sim.run_sim(n_nodes, n_turns, bound_class(host_cls, engine_cls), **kw)


def node_trace(nd):
    """The node's graph in index space (arrival order) and its call schedule as a
    list of chunk sizes (one divide_rounds call each)."""
    n = len(nd._i2h)
    p0, p1, cr, t, sig = nd._columns(list(range(n)))
    sizes = [op[2] for op in nd._ops if op[0] == "d"]
    assert sum(sizes) == n
    return Trace(len(nd._m2pk), p0, p1, cr, t, sig, "node"), sizes


def node_results(nd):
    rnd = np.array([nd.round[h] for h in nd._i2h], np.int32)
    fam = np.array([(1 if nd.famous[h] else 0) if h in nd.famous else -1 for h in nd._i2h], np.int8)
    tx = np.array([nd._h2i[h] for h in nd.transactions], np.int32)
    return {"round": rnd, "famous": fam, "transactions": tx,
            "consensus": np.array(sorted(nd.consensus), np.int32)}


def replay_oracle(tr, sizes):
    import oracle as orc
    o = orc.Oracle(tr.M)
    o.append(tr)
    first = 0
    for s in sizes:
        o.divide_rounds(first, s)
        o.find_order(o.decide_fame())
        first += s
    return o.results()


def replay_node(g, engine_cls=None):
    """A bound node fed a recorded node trace (fixture `g`: trace columns + call schedule) the way a host feeds it:
    its own root from `new_event`, then per call the new events through `add_event` and one (divide_rounds,
    decide_fame, find_order) triple.  Ids and member keys are synthetic; the engine reads parents, creator, time and
    signature only."""
    M, sizes = int(g["M"]), g["sizes"].tolist()
    pks = [bytes([m]) * 32 for m in range(M)]
    ids = [i.to_bytes(8, "little") for i in range(len(g["p0"]))]

    def event(i):
        p = () if g["p0"][i] < 0 else (ids[g["p0"][i]], ids[g["p1"][i]])
        return host_sim.Event(None, p, float(g["t"][i]), pks[g["creator"][i]], bytes(g["sig"][i]))

    class Replay:
        def new_event(self, d, p):
            return ids[0], event(0)

    assert sizes[0] == 1
    nd = bound_class(Replay, engine_cls)((pks[g["creator"][0]], b""), {}, M, {pk: 1 for pk in pks})
    first = 1
    for s in sizes[1:]:
        for i in range(first, first + s):
            nd.add_event(ids[i], event(i))
        nd.divide_rounds(ids[first:first + s])
        nd.find_order(nd.decide_fame())
        first += s
    return nd

