"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(a checkout of Lapin0t/py-swirld, imported in place through oracle/ref_harness.py)
on the traces and call schedules of oracle/golden_specs.py.

    SWIRLD_REFERENCE=<py-swirld checkout> python oracle/make_golden.py [name ...]

Each fixture holds, in index space: round[N], witness_table[R,M], famous[N]
(-1 = no entry), consensus[], transactions[], the per-call new_c lists
(flattened), sha256 of the can_see matrix (and the matrix itself when small).
"""
from __future__ import annotations

import hashlib
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "py-swirld_b200"))
sys.path.insert(0, HERE)

import golden_specs as gs  # noqa: E402
import ref_harness as rh   # noqa: E402


def fixture(tr, r):
    """The reference's results `r` on trace `tr` as the arrays of one fixture."""
    cs = rh.can_see_matrix(r["can_see_node"], tr.N, tr.M)
    flat, offs = [], [0]
    for nc in r["new_c_per_call"]:
        flat.extend(nc)
        offs.append(len(flat))
    out = dict(
        round=r["round"], witness_table=r["witness_table"], famous=r["famous"],
        consensus=r["consensus"], transactions=r["transactions"],
        new_c_flat=np.array(flat, dtype=np.int32), new_c_offs=np.array(offs, dtype=np.int32),
        can_see_sha256=np.frombuffer(hashlib.sha256(cs.tobytes()).digest(), dtype=np.uint8),
        trace_sha256=np.frombuffer(hashlib.sha256(
            tr.p0.tobytes() + tr.p1.tobytes() + tr.creator.tobytes() + tr.t.tobytes()
            + tr.sig.tobytes()).digest(), dtype=np.uint8),
        ref_seconds=np.array([r["t_divide_rounds"], r["t_decide_fame"], r["t_find_order"]]),
    )
    if cs.size <= 200000:
        out["can_see"] = cs
    return out


def main(names):
    os.makedirs(gs.GOLDEN_DIR, exist_ok=True)
    for name in names:
        tr, K, stake = gs.make_trace(name)
        t0 = time.time()
        r = rh.run_reference(tr, K, stake)
        np.savez_compressed(gs.path(name), **fixture(tr, r))
        print("%-32s N=%d M=%d K=%d  max_r=%d wit=%d famous=%d/%d cons=%d ordered=%d  "
              "ref dr=%.2fs df=%.2fs fo=%.2fs  (%.1fs, %d KB)" % (
                  name, tr.N, tr.M, K, r["round"].max(), int(r["witness"].sum()),
                  int((r["famous"] >= 0).sum()), int((r["famous"] == 1).sum()),
                  len(r["consensus"]), len(r["transactions"]),
                  r["t_divide_rounds"], r["t_decide_fame"], r["t_find_order"],
                  time.time() - t0, os.path.getsize(gs.path(name)) // 1024), flush=True)


def node_sim_fixtures():
    """gs.NODE_SIM: the arrival traces and call schedules of the first nodes of one gossip simulation (the oracle
    standing in for the engine), each with the reference's replay of it."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import node_sim
    from oracle_engine import OracleEngine
    node_fixtures(gs.NODE_SIM, node_sim.run_sim(4, 400, OracleEngine, capacity=64, seed=5))


def drop_in_fixtures():
    """gs.DROP_IN: the same for every node of the reference's own driver, swirld.test(4, 300), run over
    bind(swirld.Node) with the oracle standing in for the engine."""
    import contextlib
    import io
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import node_sim
    from oracle_engine import OracleEngine
    swirld = rh.load_reference()
    saved = swirld.Node
    try:
        swirld.Node = node_sim.bound_class(saved, OracleEngine)
        with contextlib.redirect_stdout(io.StringIO()):
            nodes = swirld.test(4, 300)
    finally:
        swirld.Node = saved
    node_fixtures(gs.DROP_IN, nodes)


def node_fixtures(names, nodes):
    import node_sim
    for name, nd in zip(names, nodes):
        tr, sizes = node_sim.node_trace(nd)
        r = rh.run_reference(tr, sizes)
        np.savez_compressed(gs.path(name), M=tr.M, p0=tr.p0, p1=tr.p1, creator=tr.creator, t=tr.t, sig=tr.sig,
                            sizes=np.array(sizes, np.int32), **fixture(tr, r))
        print("%-32s N=%d M=%d calls=%d  (%d KB)" % (name, tr.N, tr.M, len(sizes),
                                                     os.path.getsize(gs.path(name)) // 1024), flush=True)


if __name__ == "__main__":
    if not rh.reference_available():
        sys.exit("SWIRLD_REFERENCE must name a checkout of the reference (Lapin0t/py-swirld)")
    names = sys.argv[1:] or list(gs.SPECS) + list(gs.SPOTS) + gs.NODE_SIM + gs.DROP_IN
    main([n for n in names if n not in gs.NODE_SIM + gs.DROP_IN])
    if any(n in gs.NODE_SIM for n in names):
        node_sim_fixtures()
    if any(n in gs.DROP_IN for n in names):
        drop_in_fixtures()
