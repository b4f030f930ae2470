#!/usr/bin/env python
"""bench.py -- events/s through divide_rounds + decide_fame (BASELINE.json's metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c3] [--dump-outputs DIR]

A "step" is one pass of the hot path over the whole synthetic trace of the workload: for every
chunk of the pinned call schedule, `divide_rounds(chunk)` then `decide_fame()` (swirld.py:325-327),
starting from an engine whose consensus state was cleared.  Workloads (BASELINE.json `configs`):
    c1  4 members,     2 000 events, K=50        G1 (plumbing)
    c2  16 members,  100 000 events, K=4096      G1
    c3  64 members, 1 000 000 events, K=65536    G1   <- headline, default
    c4  256 members, 4 000 000 events, K=262144  G1 (vectorised generator)
    c5  1024 members, 16 000 000 events, K=262144  G2 adversarial (two cliques, p_cross 0.02, stale other-parents 0.3)
`--events` runs a prefix of the workload's event count.

`value`   : events/s with the event columns already resident in HBM (sw_rewind keeps them),
            device-timed with CUDA events on the engine's stream; max over ranks.
`e2e`     : the same metric through the C ABI from HOST buffers: every step clears the engine, appends each chunk
            from pinned host memory (H2D inside the timed region), runs divide_rounds + decide_fame per chunk and
            reads back round / witness / famous for all events (D2H inside the timed region).
`parity`  : the engine's round / witness / famous (c1-c3: of the whole trace; c4-c5: of a prefix run with the prefix
            as one chunk) compared element-wise with the oracle's, in this run.  A mismatch exits non-zero.
`roofline`: the dominant kernel of the step (M <= 64: the round kernel -- k_rounds_cluster for chunks of >= 2048
            events, k_rounds_batch below; above 64 members: k_rounds_wide or the can_see scan, whichever takes longer) -- algorithmic bytes per event (SURVEY.md section 8d) over its mean launch
            duration (CUDA events on the engine's stream) against MEASURED_PEAKS.json hbm_gbs.
`roofline_can_see`: the same for the can_see kernel family k_cs_* (B1(M) = 12M + 12 bytes per event).
`cpu_baseline` / --impl reference: the literal C restatement oracle/ (kind "port"), single-threaded per node-view
            like the reference (README.md:27-28), plus -- where SWIRLD_REFERENCE names a checkout of the reference --
            the UNMODIFIED Python reference timed on a prefix of the same trace (`python_reference`).
`--dump-outputs DIR`: what the last timed step computed (rank 0) as DIR/<name>.npy, float32 (float64 for event
            indices past 2**24 and for the sample index), at most 64 MiB in all: round, witness, famous per event --
            a fixed seeded sample of the events (sample_index.npy) when the whole columns would not fit -- and the
            witness_table and consensus rounds.  The traces are seeded, so the same arguments give the same inputs.

N > 1, one process per GPU (torchrun):
  c1-c3 (M <= 64): independent node-views ("replicas", DESIGN.md section 6: a round step costs less than any
          cross-GPU exchange), own trace per rank, no collective on the data path, scaling "weak";
  c4-c5 (M > 64): ONE hashgraph on all ranks: the P_r tests of every round step are sharded by member chain and the
          ranks write their first hits into each other's buffers over NVLink from inside k_rounds_wide
          (sw_peer_connect; handles exchanged once through torch.distributed); scaling "strong".
Ranks meet at a barrier before and after the timed region and the time is the max over ranks.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "py-swirld_b200"))

import numpy as np  # noqa: E402

WORKLOADS = {
    "c1": dict(M=4, N=2000, K=50, gen="gossip"),
    "c2": dict(M=16, N=100000, K=4096, gen="gossip"),
    "c3": dict(M=64, N=1000000, K=65536, gen="gossip"),
    "c4": dict(M=256, N=4000000, K=262144, gen="gossip_np"),
    "c5": dict(M=1024, N=16000000, K=262144, gen="adversarial_np"),
}
GEN_TEXT = {"gossip": "G1 reference-sim gossip", "gossip_np": "G1 reference-sim gossip (vectorised generator)",
            "adversarial_np": "G2 adversarial gossip (two cliques, p_cross 0.02, stale other-parents 0.3; vectorised generator)"}

# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel at c3 (65536 events), from the
# committed ncu --set full capture (profiles/README.md); None where no capture of that launch shape exists
DRAM_BYTES_PER_LAUNCH = {("k_rounds_batch", 64, 65536): 18547712 + 2816,
                         ("k_rounds_cluster", 64, 65536): 17356288 + 0}


def algorithmic_bytes_per_event(M):
    """SURVEY.md section 8d: divide_rounds + decide_fame combined."""
    return 12 * M + 12 + 5 + M / 8.0


def can_see_bytes_per_event(M):
    """SURVEY.md section 8d, K1: read two parent rows, write one, read p0/p1/creator."""
    return 12 * M + 12


def rounds_bytes_per_event(M):
    """the round kernel: read row(h), p0, creator; write round, witness flag, seen-mask."""
    return 4 * M + 8 + 5 + M / 8.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True,
                                     timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for s in self.samples for i in range(4)
                          if len(s) >= 6 and s[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def make_trace(wl, seed):
    from swirld_b200 import traces
    gen = wl.get("gen", "gossip")
    cache = os.path.join(tempfile.gettempdir(), "swirld_trace_%s_M%d_N%d_s%d.npz" % (gen, wl["M"], wl["N"], seed))
    if os.path.exists(cache):
        try:
            z = np.load(cache)
            return traces.Trace(wl["M"], z["p0"], z["p1"], z["creator"], z["t"], z["sig"], gen + " cached")
        except Exception:
            pass
    tr = getattr(traces, gen)(wl["M"], wl["N"], seed)
    if wl["N"] <= 2000000:
        try:
            tmp = cache + ".%d.tmp.npz" % os.getpid()
            np.savez(tmp, p0=tr.p0, p1=tr.p1, creator=tr.creator, t=tr.t, sig=tr.sig)
            os.replace(tmp, cache)
        except Exception:
            pass
    return tr


def sharded(wl):
    """M > 64: one hashgraph over all ranks (strong scaling); else independent node-views (weak)."""
    return wl["M"] > 64


# --------------------------------------------------------------------------- CPU arm
def run_cpu_pass(tr, K, limit=None):
    """One pass of divide_rounds + decide_fame (+ find_order, untimed) through the
    oracle port; returns (events, seconds in dr+df, seconds in find_order, results)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    n = tr.N if limit is None else min(limit, tr.N)
    res = orc.run_oracle(tr.slice(0, n), K)
    res["oracle"].close()
    return n, res["t_divide_rounds"] + res["t_decide_fame"], res["t_find_order"], res


def port_rate_guess(M):
    """events/s of the C port on one core (measured: 2.3e5 at M=64; the literal loops are O(M^2) per event)."""
    return 2.3e5 * (64.0 / max(M, 4)) ** 2 if M >= 64 else 2.3e5 * min(16.0, (64.0 / M))


def reference_sample_events(wl, steps):
    """Events per step of the CPU arm: the whole trace when the run stays within about a minute of CPU work,
    else a prefix (whole chunks where a chunk fits)."""
    budget = int(45 * port_rate_guess(wl["M"]) / max(1, steps))
    if budget >= wl["N"]:
        return wl["N"]
    if budget >= wl["K"]:
        return budget // wl["K"] * wl["K"]
    return max(2000, min(wl["K"], budget))


def python_reference_sample(tr, wl):
    """The UNMODIFIED Python reference (the checkout SWIRLD_REFERENCE names) on a prefix of the trace: events/s
    through its own divide_rounds + decide_fame.  None without one."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_harness as rh
    if not rh.reference_available():
        return None
    try:
        M = wl["M"]
        n = min(tr.N, max(2000, 3 * M, int(12 * 5.6e3 * (64.0 / max(M, 8)) ** 2)))     # ~10-40 s of CPython; past the M root events
        K = min(wl["K"], 2000) if n > 2000 else wl["K"]
        r = rh.run_reference(tr.slice(0, n), K)
        s = r["t_divide_rounds"] + r["t_decide_fame"]
        return {"value": n / s, "unit": "events/s", "cores": 1, "kind": "reference-python",
                "sample": "first %d events, K=%d, unmodified swirld.py through oracle/ref_harness.py, "
                          "divide_rounds %.2f s + decide_fame %.2f s (find_order %.2f s not counted)" % (
                              n, K, r["t_divide_rounds"], r["t_decide_fame"], r["t_find_order"])}
    except Exception as ex:      # the reference arm must not take the bench down
        return {"unavailable": "%s: %s" % (type(ex).__name__, ex)}


def _reference_replica(job):
    """One node-view through the CPU port (runs in its own process when world > 1)."""
    wl, seed, steps, warm = job
    tr = make_trace(wl, seed)
    limit = reference_sample_events(wl, steps)
    if warm:
        run_cpu_pass(tr, wl["K"], limit=min(limit, 50000))
    t0 = time.perf_counter()
    tot_e, tot_s, t_fo = 0, 0.0, 0.0
    for _ in range(steps):
        n, s, fo, _ = run_cpu_pass(tr, wl["K"], limit)
        tot_e += n
        tot_s += s
        t_fo += fo
    return tot_e, tot_s, t_fo, time.perf_counter() - t0


def bench_reference(args, wl, rank, world):
    """The CPU arm on the workload of the GPU arm.  Replica workloads (M <= 64): `world` independent node-views, one
    host core each -- the reference is single-threaded per node (README.md:27-28), so replicas are the only way it can
    use more cores.  Sharded workloads (M > 64): the GPU arm runs ONE graph however many GPUs it has, and so does
    this arm (one core: the algorithm is sequential in the events)."""
    if rank != 0:
        return
    nrep = 1 if sharded(wl) else world
    jobs = [(wl, rank_seed(r, wl), args.steps, args.warmup >= 1) for r in range(nrep)]
    if nrep == 1:
        res = [_reference_replica(jobs[0])]
    else:
        import concurrent.futures as cf
        import multiprocessing as mp
        with cf.ProcessPoolExecutor(nrep, mp_context=mp.get_context("spawn")) as ex:
            res = list(ex.map(_reference_replica, jobs))
    tot_e = sum(r[0] for r in res)
    slow = max(r[1] for r in res)                # the job is as slow as its slowest replica
    t_fo = max(r[2] for r in res)
    v = tot_e / slow
    sample = reference_sample_events(wl, args.steps)
    line = {
        "impl": "reference", "metric": "events/sec divide_rounds+decide_fame", "value": v, "unit": "events/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * slow / args.steps,
        "higher_is_better": True, "scaling": "strong" if sharded(wl) else "weak", "vs_baseline": None, "dtype": "int32",
        "data": "synthetic", "config": workload_config(wl, world),
        "cpu_baseline": {"value": v, "unit": "events/s", "cores": nrep, "kind": "port",
                         "sample": "first %d of %d events x %d passes per node-view, %d node-view(s) in parallel processes, "
                                   "oracle/swirld_oracle.c (literal C restatement of swirld.py:187-277, pinned to the "
                                   "reference by tests/golden), host has %d cpus" % (sample, wl["N"], args.steps, nrep,
                                                                                    os.cpu_count())},
        "e2e": {"value": v, "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "find_order_events_per_s": tot_e / t_fo if t_fo > 0 else None,
        "python_reference": python_reference_sample(make_trace(wl, rank_seed(0, wl)), wl),
    }
    print(json.dumps(line), flush=True)


def workload_config(wl, world):
    par = ("one hashgraph on %d GPU(s): round-step tests sharded by member chain, first hits exchanged by P2P stores "
           "over NVLink inside the round kernel" % world) if sharded(wl) else \
          ("replicas x%d (independent node-views, no collective)" % world)
    return {"workload": "%s trace, %d members x %d events, call schedule K=%d events per (divide_rounds, decide_fame) "
                        "pair, unit stake, coin period 6" % (GEN_TEXT.get(wl.get("gen", "gossip"), wl.get("gen")),
                                                            wl["M"], wl["N"], wl["K"]),
            "members": wl["M"], "events": wl["N"], "chunk": wl["K"], "parallelism": par,
            "l2": "L2 flushed (256 MiB device memset) before every timed step; the per-step working set (can_see "
                  "table) also exceeds L2 from c3 up"}


# --------------------------------------------------------------------------- streaming cadence (SURVEY.md section 8f-1)
def stream_leg(local_rank, cases=((4, 2000, 1), (4, 2000, 50), (64, 20000, 3))):
    """The reference's own cadence: one (divide_rounds, decide_fame, find_order) triple per sync, a handful of events
    per call (swirld.py:319-328).  Wall-clock through the C ABI -- sw_append + sw_divide_rounds (one launch:
    k_stream_divide) + sw_decide_fame + sw_find_order per call, from host buffers -- next to the oracle port and the
    unmodified Python reference on the SAME schedule (all three calls counted for every arm)."""
    from swirld_b200 import engine, traces
    from swirld_b200.traces import chunks
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as orc
    import ref_harness as rh
    out = []
    for M, N, K in cases:
        tr = traces.gossip(M, N, 1)
        o = orc.run_oracle(tr, K)
        t_port = o["t_divide_rounds"] + o["t_decide_fame"] + o["t_find_order"]
        best, res = None, None
        for rep_i in range(3):
            e = engine.Engine(M, N, device=local_rank)
            e.sync()
            t0 = time.perf_counter()
            ncalls = 0
            for first, cnt in chunks(N, K):
                e.append_trace(tr, first, cnt)
                e.divide_rounds(first, cnt)
                e.find_order(e.decide_fame())
                ncalls += 1
            e.sync()
            dt = time.perf_counter() - t0
            if rep_i and (best is None or dt < best):
                best = dt
            res = e.results()
            launches = e.stats()["kernel_launches"]
            e.close()
        same = all(np.array_equal(np.asarray(o[k]), np.asarray(res[k])) for k in ("round", "witness_table", "famous", "consensus", "transactions"))
        pyref = None
        if rh.reference_available():
            try:
                npre = min(N, 6000 if M >= 64 else 2000)
                r = rh.run_reference(tr.slice(0, npre), K)
                pyref = npre / (r["t_divide_rounds"] + r["t_decide_fame"] + r["t_find_order"])
            except Exception as ex:
                pyref = "unavailable: %s" % ex
        out.append({"members": M, "events": N, "events_per_call": K, "calls": ncalls,
                    "events_per_s": N / best, "us_per_call": 1e6 * best / ncalls, "kernel_launches_per_call": launches / ncalls,
                    "port_events_per_s": N / t_port, "python_reference_events_per_s": pyref, "equals_oracle": bool(same)})
        o["oracle"].close()
    return out


# --------------------------------------------------------------------------- multi-rank plumbing
def rank_seed(rank, wl=None):
    """Replica workloads: every rank advances its own node-view (an independent trace).  Sharded workloads: all
    ranks hold the same graph."""
    if wl is not None and sharded(wl):
        return 1
    return 1 + rank


def max_over_ranks(values, dist, device):
    """Element-wise max of a few per-rank timings (the job is as slow as its slowest rank)."""
    import torch
    t = torch.tensor([float(v) for v in values], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t.tolist()]


def whole_job_rate(world, events_per_rank_step, steps, ms_max, shard=False):
    """events/s of the whole job: all ranks' events over the slowest rank's time (one shared graph when sharded)."""
    return (1 if shard else world) * events_per_rank_step * steps / (ms_max * 1e-3)


def connect_peers(eng, dist, rank, world):
    """sw_peer_connect: exchange the CUDA IPC handles of the engines' exchange buffers once, out of band."""
    mine = eng.peer_handle()
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    eng.peer_connect(rank, world, b"".join(parts))


# --------------------------------------------------------------------------- output dump
DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, n_events, per_event, tables):
    """per_event: name -> column of n_events values; tables: name -> array (event indices, round numbers).  Writes
    each as out_dir/<name>.npy, float32 while event indices stay exact in it, else float64.  When the columns do not
    fit in DUMP_BYTES beside the tables, the same seeded sample of events is taken from each, its indices in
    sample_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    fdt = np.dtype(np.float32 if n_events <= 1 << 24 else np.float64)
    out = {k: np.asarray(v).astype(fdt) for k, v in tables.items()}
    room = DUMP_BYTES - (64 << 10) - sum(v.nbytes for v in out.values())      # (64 KiB for the .npy headers)
    row = len(per_event) * fdt.itemsize
    if n_events * row > room:
        keep = room // (row + 8)
        if keep < 1:
            raise SystemExit("bench.py: --dump-outputs: the tables alone exceed %d bytes" % DUMP_BYTES)
        idx = np.sort(np.random.default_rng(20240917).choice(n_events, keep, replace=False))
        out["sample_index"] = idx.astype(np.float64)
        per_event = {k: np.asarray(v)[idx] for k, v in per_event.items()}
    out.update({k: np.asarray(v).astype(fdt) for k, v in per_event.items()})
    for k, v in out.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# --------------------------------------------------------------------------- GPU arm
def bench_ours(args, wl, rank, world, local_rank):
    import torch
    from swirld_b200 import engine
    from swirld_b200.traces import chunks
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    M, N, K = wl["M"], wl["N"], wl["K"]
    shard = sharded(wl)
    tr = make_trace(wl, rank_seed(rank, wl))
    # pinned host copies of the event columns (the e2e leg's source)
    pin = {}
    for k in ("p0", "p1", "creator", "t", "sig"):
        src = torch.from_numpy(np.ascontiguousarray(getattr(tr, k)))
        pin[k] = src.pin_memory().numpy()
    out_round = torch.empty(N, dtype=torch.int32).pin_memory().numpy()
    out_wit = torch.empty(N, dtype=torch.uint8).pin_memory().numpy()
    out_fam = torch.empty(N, dtype=torch.int8).pin_memory().numpy()

    eng = engine.Engine(M, N, device=local_rank)
    if shard and world > 1:
        connect_peers(eng, dist, rank, world)
    sched = list(chunks(N, K))

    def append_all():
        for first, cnt in sched:
            s = slice(first, first + cnt)
            eng.append(pin["p0"][s], pin["p1"][s], pin["creator"][s], pin["t"][s], pin["sig"][s])

    timed_launches = [0]

    def step_resident():
        eng.rewind()
        eng.flush_l2()
        l0 = eng.stats()["kernel_launches"]       # (syncs; before the timed region)
        if dist is not None and shard:
            dist.barrier()                        # the ranks of one graph enter the step together
        eng.record(0)
        for first, cnt in sched:
            eng.divide_rounds(first, cnt)
            eng.decide_fame()
        eng.record(1)
        ms = eng.elapsed_ms(0, 1)
        timed_launches[0] += eng.stats()["kernel_launches"] - l0
        return ms

    def step_e2e():
        eng.reset()
        eng.flush_l2()
        eng.sync()
        if dist is not None and shard:
            dist.barrier()
        t0 = time.perf_counter()

        def feed(i):
            first, cnt = sched[i]
            s = slice(first, first + cnt)
            eng.append(pin["p0"][s], pin["p1"][s], pin["creator"][s], pin["t"][s], pin["sig"][s])

        # the caller's software pipeline: appends run two chunks ahead of the consensus calls (sw_append: host
        # checks, asynchronous H2D and the can_see scan of the new events on the engine's copy stream), so
        # they overlap the round kernels of earlier chunks; sw_decide_fame is the synchronising call
        ahead = 2
        for i in range(min(ahead, len(sched))):
            feed(i)
        for i, (first, cnt) in enumerate(sched):
            eng.divide_rounds(first, cnt)
            if i + ahead < len(sched):
                feed(i + ahead)
            eng.decide_fame()
        lib, h = eng._lib, eng._h
        lib.sw_get_round(h, 0, N, out_round.ctypes.data_as(C.c_void_p))
        lib.sw_get_witness_flags(h, 0, N, out_wit.ctypes.data_as(C.c_void_p))
        lib.sw_get_famous(h, 0, N, out_fam.ctypes.data_as(C.c_void_p))
        eng.sync()
        return (time.perf_counter() - t0) * 1e3

    # ---- resident-input leg (the contract's timed region)
    append_all()
    for _ in range(args.warmup):
        step_resident()
    st0 = eng.stats()
    timed_launches[0] = 0
    barrier()
    with ClockSampler(local_rank) as clk:
        t0 = time.perf_counter()
        dev_ms = 0.0
        for _ in range(args.steps):
            dev_ms += step_resident()
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
        barrier()
    st1 = eng.stats()
    got_round, got_wit, got_fam = eng.rounds(), eng.witness_flags(), eng.famous()
    check = (int(got_round.astype(np.int64).sum()), int(eng.max_round), int(len(eng.consensus())))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, N, {"round": got_round, "witness": got_wit, "famous": got_fam},
                     {"witness_table": eng.witness_table(), "consensus": eng.consensus()})

    # ---- several node-views per launch (M <= 64: SURVEY.md section 8f-3): B independent views (own traces) advanced by
    #      sw_batch_divide_rounds, aggregate events/s over all views, device-timed on the first view's stream
    views_out = None
    if args.views and not shard and M <= 64:
        views_out = []
        Nv = min(N, args.views_events) if args.views_events else N
        for B in [int(x) for x in args.views.split(",")]:
            trs = [make_trace(dict(wl, N=Nv, gen="gossip_np"), 1000 + 17 * rank + v) for v in range(B)]   # (vectorised generator: B traces)
            engs = [engine.Engine(M, Nv, device=local_rank) for _ in range(B)]
            for ev, tv in zip(engs, trs):
                ev.append_trace(tv)
            vs = list(chunks(Nv, K))
            best = None
            for rep_i in range(1 + max(1, args.steps // 4)):
                for ev in engs:
                    ev.rewind()
                torch.cuda.synchronize()
                t0v = time.perf_counter()
                for first, cnt in vs:
                    engine.batch_divide_rounds(engs, [first] * B, [cnt] * B)
                    for ev in engs:
                        ev.decide_fame()
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0v
                if rep_i and (best is None or dt < best):      # (the first pass is the warm-up)
                    best = dt
            ok_v = True
            if B <= 8:
                ov = run_cpu_pass(trs[-1], K)[3]
                ok_v = bool(np.array_equal(ov["round"], engs[-1].rounds()) and np.array_equal(ov["famous"], engs[-1].famous()))
            views_out.append({"views": B, "events_per_view": Nv, "events_per_s": B * Nv / best, "ms": best * 1e3,
                              "last_view_equals_oracle": ok_v})
            for ev in engs:
                ev.close()

    # ---- find_order, timed separately (not part of the metric); every rank runs it (replicated)
    fo_ms, n_ordered = None, None
    if not args.no_find_order and M <= 256:
        eng.rewind()
        fo_ms0 = eng.stats()["ms_find_order"]
        for first, cnt in sched:
            eng.divide_rounds(first, cnt)
            eng.find_order(eng.decide_fame())
        fo_ms = eng.stats()["ms_find_order"] - fo_ms0
        n_ordered = eng.n_transactions

    # ---- end-to-end leg from host buffers
    for _ in range(min(args.warmup, 2)):
        step_e2e()
    barrier()
    e2e_ms = 0.0
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        e2e_ms += step_e2e()
    st_e2e = eng.stats()              # sw_reset clears the counters: this is the last e2e step alone
    e2e_same = bool(np.array_equal(out_round, got_round) and np.array_equal(out_wit, got_wit) and np.array_equal(out_fam, got_fam))
    barrier()

    dev_ms_max, e2e_ms_max, wall_ms_max = max_over_ranks([dev_ms, e2e_ms, wall_ms], dist, "cuda")
    # sharded: every rank must hold identical results
    same_on_all = True
    if dist is not None and shard:
        digest = torch.tensor([check[0], check[1], check[2], int(got_fam.astype(np.int64).sum()), int(got_wit.sum())],
                              dtype=torch.int64, device="cuda")
        lo, hi = digest.clone(), digest.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        same_on_all = bool(torch.equal(lo, hi))

    ok = True
    if rank == 0:
        peak, peak_src = load_peaks()
        launches = timed_launches[0]
        ms_div = st1["ms_divide_rounds"] - st0["ms_divide_rounds"]
        ms_fame = st1["ms_decide_fame"] - st0["ms_decide_fame"]
        n_div_launch = len(sched) * args.steps
        ms_cs = st1["ms_can_see"] - st0["ms_can_see"]
        ms_rk = st1["ms_rounds_kernel"] - st0["ms_rounds_kernel"]
        wide = M > 64 or os.environ.get("SW_FORCE_WIDE", "0") not in ("", "0")
        cluster = (not wide and K >= int(os.environ.get("SW_RC_MIN_N", "2048"))
                   and os.environ.get("SW_ROUNDS_CLUSTER", "1") not in ("", "0"))
        rk_name = "k_rounds_wide" if wide else ("k_rounds_cluster" if cluster else "k_rounds_batch")
        dominant_cs = ms_cs > ms_rk
        cs_achieved = (N * args.steps * can_see_bytes_per_event(M)) / (ms_cs * 1e-3) / 1e9 if ms_cs > 0 else None
        rk_achieved = (N * args.steps * rounds_bytes_per_event(M)) / (ms_rk * 1e-3) / 1e9 if ms_rk > 0 else None
        path_achieved = (N * args.steps * algorithmic_bytes_per_event(M)) / ((ms_div + ms_fame) * 1e-3) / 1e9
        value = whole_job_rate(world, N, args.steps, dev_ms_max, shard)
        e2e_value = whole_job_rate(world, N, e2e_steps, e2e_ms_max, shard)
        # ---- parity + CPU baseline next to it: the oracle port on the box's host cores, in this run
        if N * (M / 64.0) ** 2 <= 1.2e6:
            n_cpu, s_cpu, fo_cpu, ores = run_cpu_pass(tr, K)
            exp_wit = np.zeros(N, np.uint8)
            wt = ores["witness_table"]
            exp_wit[wt[wt >= 0]] = 1
            par = {"scope": "all %d events, element-wise" % N,
                   "round": bool(np.array_equal(ores["round"], got_round)),
                   "witness": bool(np.array_equal(exp_wit, got_wit)),
                   "famous": bool(np.array_equal(ores["famous"], got_fam))}
            cpu_sample = "full trace (%d events)" % n_cpu
        else:
            npre = max(2000, 3 * M, min(N, int((30 if world == 1 else 10) * port_rate_guess(M))))   # (the other ranks wait: keep it short)
            n_cpu, s_cpu, fo_cpu, ores = run_cpu_pass(tr, npre, limit=npre)
            e2 = engine.Engine(M, npre, device=local_rank)
            e2.append_trace(tr, 0, npre)
            e2.divide_rounds(0, npre)
            e2.decide_fame()
            exp_wit = np.zeros(npre, np.uint8)
            wt = ores["witness_table"]
            exp_wit[wt[wt >= 0]] = 1
            par = {"scope": "prefix of %d events as one chunk (the literal oracle is O(M^2) per event), element-wise; "
                            "full length: identical on all ranks = %s" % (npre, same_on_all),
                   "round": bool(np.array_equal(ores["round"], e2.rounds())),
                   "witness": bool(np.array_equal(exp_wit, e2.witness_flags())),
                   "famous": bool(np.array_equal(ores["famous"], e2.famous())),
                   "can_see": bool(np.array_equal(ores["oracle_can_see"], e2.can_see())) if "oracle_can_see" in ores else None}
            e2.close()
            cpu_sample = "first %d events as one chunk" % n_cpu
        par["e2e_results_equal_resident"] = e2e_same
        par["identical_on_all_ranks"] = same_on_all
        ok = all(v for k, v in par.items() if k not in ("scope", "can_see") and v is not None)
        par["ok"] = ok
        dom_ms = ms_cs if dominant_cs else ms_rk
        dom_bpe = can_see_bytes_per_event(M) if dominant_cs else rounds_bytes_per_event(M)
        dom_ach = cs_achieved if dominant_cs else rk_achieved
        dom_name = "k_cs_pass<2> (can_see scan family k_cs_*)" if dominant_cs else rk_name
        line = {
            "metric": "events/sec divide_rounds+decide_fame", "value": value, "unit": "events/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if shard else "weak",
            "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": workload_config(wl, world),
            "clocks": clk.summary(),
            "parity": ok, "parity_detail": par,
            "e2e": {"value": e2e_value, "unit": "events/s",
                    # counted by the library from the copies it issued in the last step (event columns incl. the
                    # derived seq/height/stale columns; results + per-call scalars)
                    "h2d_bytes_per_step": int(st_e2e["h2d_bytes"]), "d2h_bytes_per_step": int(st_e2e["d2h_bytes"]),
                    "ms_per_step": e2e_ms_max / e2e_steps,
                    "kernel_ms_last_step": {"divide_rounds": st_e2e["ms_divide_rounds"], "can_see_scan": st_e2e["ms_can_see"],
                                            "rounds_kernel": st_e2e["ms_rounds_kernel"], "decide_fame": st_e2e["ms_decide_fame"]},
                    "what": "reset + per chunk: sw_append (host checks, pinned host -> HBM) + sw_divide_rounds + "
                            "sw_decide_fame, appends issued two chunks ahead of the consensus calls so that the copies "
                            "and the can_see scan overlap the round kernels; then round/witness/famous of every event "
                            "back to pinned host"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom_name,
                         "achieved": dom_ach, "peak": peak, "unit": "GB/s", "frac": dom_ach / peak if dom_ach else None,
                         "traffic": DRAM_BYTES_PER_LAUNCH.get((rk_name, M, K)) if not dominant_cs else None,
                         "traffic_source": "ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one launch "
                                           "(profiles/README.md)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_event": dom_bpe, "events_per_launch": K,
                         "ms_per_launch": dom_ms / n_div_launch,
                         "note": "latency-bound, not HBM-bound: the depth of the computation is the number of rounds (one step "
                                 "per round at M <= 64 -- inside one thread-block cluster for chunks >= 2048 events, "
                                 "grid-wide below --, a few grid-wide steps per round above 64 members); ms_per_launch "
                                 "covers the round kernel(s) of one divide_rounds call (k_rc_seqrows + k_rounds_cluster "
                                 "+ the hand-over launch of k_rounds_batch); DESIGN.md section 5"},
            "roofline_can_see": None if cs_achieved is None else {
                "bound": "hbm", "kernel": "k_cs_prep + k_cs_pass<1> + k_cs_heads + k_cs_check + k_cs_slow + k_cs_pass<2> "
                                          "(column-tiled blocked max-plus scan)",
                "achieved": cs_achieved, "peak": peak, "unit": "GB/s", "frac": cs_achieved / peak,
                "algorithmic_bytes_per_event": can_see_bytes_per_event(M), "ms_per_step": ms_cs / args.steps,
                "note": "the resident leg scans all appended events in the first divide_rounds call of a step (the "
                        "end-to-end leg scans chunk by chunk, beside the round kernel of the previous chunk)"},
            "roofline_rounds": None if rk_achieved is None else {
                "bound": "hbm", "kernel": rk_name, "achieved": rk_achieved, "peak": peak, "unit": "GB/s",
                "frac": rk_achieved / peak, "algorithmic_bytes_per_event": rounds_bytes_per_event(M),
                "ms_per_launch": ms_rk / n_div_launch},
            "roofline_path": {"bound": "hbm", "what": "all kernels of divide_rounds + decide_fame, SURVEY.md 8d B(M)",
                              "achieved": path_achieved, "peak": peak, "unit": "GB/s", "frac": path_achieved / peak,
                              "algorithmic_bytes_per_event": algorithmic_bytes_per_event(M)},
            "kernel_ms_per_step": {"divide_rounds": ms_div / args.steps, "decide_fame": ms_fame / args.steps,
                                   "can_see_scan": ms_cs / args.steps, "rounds_kernel": ms_rk / args.steps,
                                   "wall": wall_ms_max / args.steps},
            "impl": {"rounds": rk_name, "can_see": "k_cs_* column-tiled scan"},
            "cpu_baseline": {"value": n_cpu / s_cpu, "unit": "events/s", "cores": 1, "kind": "port",
                             "sample": "%s, oracle/swirld_oracle.c single thread on a host with %d cpus" % (cpu_sample, os.cpu_count())},
            "python_reference": python_reference_sample(tr, wl) if not args.no_python_reference else None,
            "find_order": None if fo_ms is None else {
                "events_per_s": n_ordered / (fo_ms * 1e-3) if fo_ms > 0 else None, "ordered": int(n_ordered),
                "ms": fo_ms, "cpu_port_events_per_s": n_cpu / fo_cpu if fo_cpu > 0 else None},
            "checksum": {"round_sum": check[0], "max_round": check[1], "consensus_rounds": check[2]},
            "views": views_out,
            "stream": stream_leg(local_rank) if args.stream else None,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--events", type=int, default=0, help="override the workload's event count")
    ap.add_argument("--no-find-order", action="store_true")
    ap.add_argument("--stream", action="store_true", help="add the streaming-cadence leg (one sync per call)")
    ap.add_argument("--views", default="", help="comma list of view counts B for the multi-view leg (M <= 64), e.g. 1,8,32")
    ap.add_argument("--views-events", type=int, default=0, help="events per view in the multi-view leg (default: the workload's)")
    ap.add_argument("--no-python-reference", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (at most 64 MiB)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the GPU arm computed; --impl reference has no such step")
    wl = dict(WORKLOADS[args.workload])
    if args.events:
        wl["N"] = args.events
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        bench_reference(args, wl, rank, world)
    else:
        bench_ours(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
