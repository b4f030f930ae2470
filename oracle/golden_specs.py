"""Trace + call-schedule specs of the committed golden fixtures (tests/golden).
Shared by oracle/make_golden.py (which runs the unmodified reference on them)
and by the tests (which rebuild the same trace and compare)."""
from __future__ import annotations

import os

SPECS = {
    # name: (generator, kwargs, K, stake or None)
    # config 1 of BASELINE.json: 4-member 2000-event gossip, the sim's cadence K=1
    "g1_m4_n2000_s1_k1":    ("gossip", dict(M=4, N=2000, seed=1), 1, None),
    "g1_m4_n2000_s1_k50":   ("gossip", dict(M=4, N=2000, seed=1), 50, None),
    "g1_m4_n2000_s1_k2000": ("gossip", dict(M=4, N=2000, seed=1), 2000, None),
    "g1_m4_n2000_s2_k1":    ("gossip", dict(M=4, N=2000, seed=2), 1, None),
    "g1_m4_n2000_s2_k50":   ("gossip", dict(M=4, N=2000, seed=2), 50, None),
    "g1_m4_n2000_s3_k7":    ("gossip", dict(M=4, N=2000, seed=3), 7, None),
    "g1_m4_n2000_s3_k2000": ("gossip", dict(M=4, N=2000, seed=3), 2000, None),
    "g1_m7_n3000_s5_k37":   ("gossip", dict(M=7, N=3000, seed=5), 37, None),
    # integer stakes (stake dict of swirld.py:42); the first never leaves round 0
    # because promotion compares a member COUNT with the STAKE threshold (quirk Q3)
    "g1_m5_n1500_s4_k11_stake": ("gossip", dict(M=5, N=1500, seed=4), 11, [1, 2, 3, 1, 2]),
    "g1_m7_n3000_s4_k11_stake": ("gossip", dict(M=7, N=3000, seed=4), 11, [1, 1, 2, 1, 1, 1, 0]),
    "g1_m10_n3000_s4_k64_stake": ("gossip", dict(M=10, N=3000, seed=4), 64, [1, 1, 1, 1, 1, 1, 1, 1, 2, 0]),
    "g2_m8_n6000_s2_k1":    ("adversarial", dict(M=8, N=6000, seed=2, p_cross=0.05, p_stale=0.3), 1, None),
    "g1_m16_n20000_s1_k1000": ("gossip", dict(M=16, N=20000, seed=1), 1000, None),
    "g2_m16_n12000_s1_k500":  ("adversarial", dict(M=16, N=12000, seed=1, p_cross=0.02, p_stale=0.3), 500, None),
    "g1_m16_n8000_s1_tied8_k1000": ("gossip", dict(M=16, N=8000, seed=1, tied=8), 1000, None),
    "g3_m16_n6000_s1_k700": ("tick", dict(M=16, N=6000, seed=1), 700, None),
    "g3_m32_n8000_s2_k512": ("tick", dict(M=32, N=8000, seed=2), 512, None),
    "g1_m33_n6000_s7_k640": ("gossip", dict(M=33, N=6000, seed=7), 640, None),
    "g2_m64_n16000_s3_k4096": ("adversarial", dict(M=64, N=16000, seed=3, p_cross=0.03, p_stale=0.3), 4096, None),
    "g1_m64_n20000_s1_k2000": ("gossip", dict(M=64, N=20000, seed=1), 2000, None),
    # config 2 of BASELINE.json in full, config 3 as a prefix (same K as the bench)
    "g1_m16_n100000_s1_k4096": ("gossip", dict(M=16, N=100000, seed=1), 4096, None),
    "g1_m64_n131072_s1_k65536": ("gossip", dict(M=64, N=131072, seed=1), 65536, None),
    # beyond 64 members (multi-word member masks): prefixes of BASELINE.json's configs 4 and 5 and mid sizes
    "g1_m96_n20000_s3_k3000": ("gossip", dict(M=96, N=20000, seed=3), 3000, None),
    "g1_m80_n8000_s4_k999_stake": ("gossip", dict(M=80, N=8000, seed=4), 999, [1 + (i % 3 == 0) for i in range(80)]),
    "g2_m128_n40000_s2_k8192": ("adversarial", dict(M=128, N=40000, seed=2, p_cross=0.02, p_stale=0.3), 8192, None),
    "g3_m128_n12000_s1_k2048": ("tick", dict(M=128, N=12000, seed=1), 2048, None),
    "g1_m256_n60000_s1_k16384": ("gossip", dict(M=256, N=60000, seed=1), 16384, None),
    "g1_m1024_n20000_s1_k8192": ("gossip", dict(M=1024, N=20000, seed=1), 8192, None),
    # a member whose root arrives ~48 rounds late (its chain starts further behind than the round kernels' mirror)
    "g4_m9_n6000_join3000_s77_k2500": ("late_joiner", dict(M=9, N=6000, join_at=3000, seed=77), 2500, None),
}


# small spot checks of the oracle against the reference (tests/test_oracle_golden.py): for each (M, N, K, seed)
# one gossip trace and one adversarial trace with at least four members
SPOT_CASES = [(4, 600, 1, 11), (5, 900, 13, 12), (16, 3000, 250, 13)]


def spot_names(M, N, K, seed):
    return ["spot_g1_m%d_n%d_s%d_k%d" % (M, N, seed, K), "spot_g2_m%d_n%d_s%d_k%d" % (max(M, 4), N, seed, K)]


SPOTS = {}
for _M, _N, _K, _seed in SPOT_CASES:
    _g1, _g2 = spot_names(_M, _N, _K, _seed)
    SPOTS[_g1] = ("gossip", dict(M=_M, N=_N, seed=_seed), _K, None)
    SPOTS[_g2] = ("adversarial", dict(M=max(_M, 4), N=_N, seed=_seed, p_cross=0.05, p_stale=0.3), _K, None)

# node traces recorded from one gossip simulation of tests/node_sim.py (4 nodes, 400 turns, seed 5: real keys and
# clock timestamps, so the traces themselves are stored), replayed through the reference with each node's own
# call schedule
NODE_SIM = ["node_sim_n4_t400_node0", "node_sim_n4_t400_node1"]
# the same for every node of one run of the reference's own driver, swirld.test(4, 300), over bind(swirld.Node)
DROP_IN = ["drop_in_n4_t300_node%d" % i for i in range(4)]

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                          "tests", "golden")


def make_trace(name):
    from swirld_b200 import traces
    gen, kw, K, stake = SPECS[name] if name in SPECS else SPOTS[name]
    return getattr(traces, gen)(**kw), K, stake


def path(name):
    return os.path.join(GOLDEN_DIR, name + ".npz")
