/*
 * swirld_b200.h -- C ABI of libswirld_b200.so, the B200 (sm_100a) engine for
 * py-swirld's consensus hot path.
 *
 * The reference (Lapin0t/py-swirld) has no FFI: its "operator interface" for this
 * path is the method surface of `swirld.Node` (/root/reference/swirld.py).  Each
 * entry point below replaces one of those methods / attributes; the Python class
 * `swirld_b200.node.GpuNode` binds them with ctypes and presents the reference's
 * own names (see INTEGRATION.md).  Index space: an event is its arrival index at
 * this node-view (int32, topological), a member is 0..M-1.
 *
 * Conventions: plain pointers and sizes only; every pointer argument is HOST
 * memory owned by the caller; device memory is owned by the engine; one CUDA
 * stream per engine; one caller thread per engine (the reference is single
 * threaded: README.md:27-28).  Functions return >= 0 on success and a negative
 * SW_E_* code on failure; sw_last_error() gives the text.  There is NO CPU
 * fallback: without a CUDA device sw_create fails with SW_E_CUDA.
 */
#ifndef SWIRLD_B200_H
#define SWIRLD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SW_OK            0
#define SW_E_ARG        -1   /* bad argument */
#define SW_E_INDEX      -2   /* reference would raise IndexError (swirld.py:305, one seer) */
#define SW_E_KEY        -3   /* reference would raise KeyError (unknown event / round) */
#define SW_E_CUDA       -4   /* CUDA runtime error or no device */
#define SW_E_CAPACITY   -5   /* capacity_events / round table exhausted */
#define SW_E_PARENT     -6   /* invalid parents: is_valid_event would be False (swirld.py:104-108) */
#define SW_E_FORK       -7   /* self-parent is not the creator's latest event (fork; swirld.py:110-112 TODO) */
#define SW_E_UNSUPPORTED -8  /* e.g. M above the compiled kernels' limit */

#define SW_MAX_MEMBERS  1024 /* member sets are ceil(M/32)-word masks; above 64 members the swirld_wide.cuh kernels run */

typedef struct sw_engine sw_engine;

/* Cumulative counters since sw_create / sw_reset (device times from CUDA events
 * recorded on the engine's stream around the kernels of each call). */
typedef struct sw_stats_t {
    double ms_divide_rounds;   /* every kernel of sw_divide_rounds (can_see scan, rounds, witnesses, k_strong) */
    double ms_decide_fame;     /* k_fame_* */
    double ms_find_order;      /* k_order_* */
    double ms_can_see;         /* subset of ms_divide_rounds spent in a stand-alone can_see kernel, 0 if fused */
    int64_t kernel_launches;   /* kernels of this library launched */
    int64_t h2d_bytes;
    int64_t d2h_bytes;
    int64_t events;            /* events appended */
    int64_t events_divided;    /* events through divide_rounds */
    double ms_rounds_kernel;   /* subset of ms_divide_rounds spent in the round-number kernel itself
                                  (M <= 64: k_rc_seqrows + k_rounds_cluster + k_rounds_batch; above: k_rounds_wide) */
} sw_stats_t;

/* Node.__init__ state (swirld.py:38-72): M members, integer stake per member
 * (NULL = unit stake as in both reference drivers, swirld.py:334 / viz.py:36),
 * coin period C (swirld.py:17), room for capacity_events events. */
int sw_create(int M, int capacity_events, const int64_t *stake, int coin_period,
              int device, sw_engine **out);
void sw_destroy(sw_engine *e);
/* Forget every event and all consensus state; keeps the allocations. */
int sw_reset(sw_engine *e);
/* Forget the consensus state (rounds, witnesses, fame, order) but keep the appended
 * event columns resident on the device: the next sw_divide_rounds starts at 0 again. */
int sw_rewind(sw_engine *e);
const char *sw_last_error(const sw_engine *e);   /* e may be NULL: last create error */

/* Node.add_event (swirld.py:114-120) for n events in arrival order, SoA columns:
 * p0/p1 = self/other parent index (-1,-1 for a root: ev.p == ()), creator,
 * t = Event.t (swirld.py:91), sig = Event.s, 64 bytes each (swirld.py:92).
 * Checks what is_valid_event checks on the graph shape (swirld.py:104-108) and
 * the fork-free contract; copies the columns to the device and, for a batch of 4096
 * events or more, starts their can_see rows (swirld.py:203-205, 220) right away.  Both run
 * on the engine's copy stream beside the kernels of earlier calls (a caller that appends a
 * chunk or two ahead of its sw_divide_rounds calls hides them completely): when the columns are in
 * page-locked host memory they must stay unchanged until the next synchronising call
 * (sw_decide_fame, sw_find_order, sw_sync, any sw_get_*); pageable memory is staged
 * before the call returns. */
int sw_append(sw_engine *e, int n, const int32_t *p0, const int32_t *p1,
              const int32_t *creator, const double *t, const uint8_t *sig);

/* Node.divide_rounds(events) (swirld.py:187-222) for the topologically sorted
 * events [first, first+n): can_see rows, round numbers, witness registration.
 * `first` must equal the number of events already divided. Asynchronous. */
int sw_divide_rounds(sw_engine *e, int first, int n);

/* Node.divide_rounds for B independent node-views in one call (the simulation's M nodes each recompute consensus on
 * nearly the same graph, swirld.py:331-345 / viz.py:35-46): engines[v] divides its events [first[v], first[v]+n[v]).
 * M <= 64, same member count and stake shape, same device.  The views' round kernels advance side by side -- one
 * thread-block cluster per view (chunks of >= 2048 events), then ONE cooperative launch, each view on its own group of
 * CTAs, for what is left: the path is latency-bound, so this is what fills the GPU.
 * Results per view are identical to B separate sw_divide_rounds calls. */
int sw_batch_divide_rounds(sw_engine *const *engines, int B, const int *first, const int *n);

/* Node.decide_fame() (swirld.py:224-277).  Writes the new consensus rounds
 * (ascending) to new_c_out[0..cap) and returns their count. */
int sw_decide_fame(sw_engine *e, int32_t *new_c_out, int cap);

/* Node.find_order(new_c) (swirld.py:280-311).  Returns the number of events
 * appended to the consensus order by this call (the caller owns the print of
 * swirld.py:310-311). */
int sw_find_order(sw_engine *e, const int32_t *new_c, int n);

/* ---- views of the Node attributes (swirld.py:48-72) ---- */
int sw_members(const sw_engine *e);           /* n (swirld.py:40) */
int sw_n_events(const sw_engine *e);          /* len(hg) */
int sw_n_divided(const sw_engine *e);         /* len(round) */
int sw_max_round(sw_engine *e);               /* max(witnesses), -1 if none */
int sw_n_transactions(const sw_engine *e);    /* len(transactions) */
int sw_get_round(sw_engine *e, int first, int n, int32_t *out);          /* round[h] */
int sw_get_witness_flags(sw_engine *e, int first, int n, uint8_t *out);  /* h in witnesses[round[h]].values() */
int sw_get_famous(sw_engine *e, int first, int n, int8_t *out);          /* famous.get(h): -1 absent, 0, 1 */
int sw_get_can_see(sw_engine *e, int first, int n, int32_t *out);        /* can_see[h] as n x M, -1 absent */
int sw_get_witness_table(sw_engine *e, int first_round, int n_rounds, int32_t *out); /* witnesses[r][c], -1 absent */
int sw_get_consensus(sw_engine *e, int32_t *out, int cap);               /* sorted(consensus) -> count */
int sw_get_transactions(sw_engine *e, int first, int n, int32_t *out);   /* transactions[first:first+n] */
int sw_get_idx(sw_engine *e, int first, int n, int32_t *out);            /* idx.get(h, -1) */
int sw_get_height(sw_engine *e, int first, int n, int32_t *out);         /* height[h] (swirld.py:68) */

int sw_sync(sw_engine *e);                     /* wait for the stream, fold timings into stats */
int sw_stats(sw_engine *e, sw_stats_t *out);   /* implies sw_sync */
/* Write >= bytes of device memory (evicts L2) on the engine's stream; for benchmarks. */
int sw_flush_l2(sw_engine *e, int64_t bytes);
/* CUDA events on the engine's stream, slots 0..15: record, and elapsed ms between two
 * recorded slots (synchronises on the later one). */
int sw_event_record(sw_engine *e, int slot);
int sw_event_elapsed_ms(sw_engine *e, int slot_a, int slot_b, double *ms_out);

/* Profiling aid: 16 cycle counters of the round kernels (tools/rounds_cycles.py). */
int sw_debug_counters(sw_engine *e, int64_t *out16, int clear);

/* ---- ingest: the step of Node.sync between the wire and divide_rounds (swirld.py:129-136, utils.py:8-21) in C++.
 * A batch of n events named by their 32-byte ids (BLAKE2b, swirld.py:95), parents given by id (32 zero bytes = none: a
 * root).  Ids the engine knows already are skipped; the others are put in a parents-first order (iterative DFS over the
 * batch; a cycle returns SW_E_ARG like toposort's ValueError), validated like sw_append validates (unknown parent,
 * parent shape, fork -- such an event, and whatever depends on it, is skipped: index -1), appended by ONE sw_append in
 * that order and entered in the engine's id -> index map.  index_out[i] = arrival index of input event i.  Returns
 * the number of events appended.  Signature and id checks are left to the caller: sw_ingest_verified makes them. */
int sw_ingest(sw_engine *e, int n, const uint8_t *ids, const uint8_t *p0_ids, const uint8_t *p1_ids,
              const int32_t *creator, const double *t, const uint8_t *sig, int32_t *index_out);
int sw_lookup(sw_engine *e, int n, const uint8_t *ids, int32_t *index_out);   /* id -> arrival index, -1 unknown */

/* ---- is_valid_event's crypto checks (swirld.py:97-103) on the GPU.
 * Public keys of the M members, 32 bytes each, in member order (Event.c; the stake dict's keys).  Decoded and checked
 * once; tables for verification (48 KB per member) built on the device.  Returns the number of members whose key
 * libsodium would reject (small order, non-canonical, not on the curve): no signature by such a member ever verifies.
 * Keys survive sw_reset / sw_rewind; they are not part of the sw_save file (call again after sw_load). */
int sw_set_member_keys(sw_engine *e, const uint8_t *pk);

/* The two checks for n events:
 *  msg  = concatenated dumps(ev[:-1]) (the signed bytes), msg_off[n+1] int64 offsets (event i: [msg_off[i], msg_off[i+1]));
 *  wire = concatenated dumps(ev)      (the hashed bytes), wire_off[n+1];
 *  sig  = n x 64 (Event.s), ids = n x 32, creator = member index.
 * status_out[i]: bit 0 = crypto_sign_verify_detached(sig, msg, pk[creator]) succeeds (libsodium's verdict exactly);
 * bit 1 = BLAKE2b-256(wire) == ids[i].  A creator outside [0, M) gives bit 0 = 0.  The engine checks the 64 bytes of
 * `sig` -- the column sw_append stores, which the coin and the whitening read; the caller is responsible for msg and
 * wire being the serialisation of that same event.  Changes no engine state.  SW_E_ARG before sw_set_member_keys.
 * Returns the number of events with status 3. */
int sw_verify(sw_engine *e, int n, const int32_t *creator, const uint8_t *sig, const uint8_t *msg, const int64_t *msg_off,
              const uint8_t *ids, const uint8_t *wire, const int64_t *wire_off, uint8_t *status_out);

/* sw_ingest with the crypto checks of is_valid_event: the new events of the batch (ids the engine does not know) are
 * verified first; one whose status is not 3 is rejected like a shape- or fork-invalid one -- index -1, and everything
 * that hangs below it is rejected too (swirld.py:133-136).  Columns as in sw_ingest and sw_verify. */
int sw_ingest_verified(sw_engine *e, int n, const uint8_t *ids, const uint8_t *p0_ids, const uint8_t *p1_ids,
                       const int32_t *creator, const double *t, const uint8_t *sig, const uint8_t *msg,
                       const int64_t *msg_off, const uint8_t *wire, const int64_t *wire_off, int32_t *index_out);

/* ---- checkpoint / resume (the reference keeps its state in memory only and uses pickle on the wire, swirld.py:129,160):
 * the engine's whole state -- event columns, can_see table, rounds, witness / fame tables, order -- as one binary file
 * of SoA sections.  sw_load builds a new engine from it (capacity_events 0 = the saved capacity; never less than the
 * saved event count) that continues exactly where the saved one stopped: the same later calls give the same results. */
int sw_save(sw_engine *e, const char *path);
int sw_load(const char *path, int device, int capacity_events, sw_engine **out);

/* ---- several GPUs of one box (one process per GPU), M > 64: ONE hashgraph, identical state and results on every rank,
 * no collective library call on the data path (the reference has no counterpart: it is single-process, swirld.py:331-345):
 *  - can_see: the column tiles of the scan are split over the ranks and every walk stores its row segments straight into
 *    EVERY rank's table over NVLink (P2P stores: the all-gather of the table is fused into the kernel that produces it);
 *  - divide_rounds: the P_r tests of every round step are sharded by member chain; every rank writes its chains' first
 *    hits into every peer's exchange buffer (P2P stores + a system-scope flag) from inside the round kernel.
 * sw_peer_handle writes SW_PEER_HANDLE_BYTES bytes (the CUDA IPC handles of this engine's exchange buffer and can_see
 * table); exchange them out of band (torch.distributed.all_gather_object), then
 * sw_peer_connect(rank, nranks <= 8, handles[nranks][SW_PEER_HANDLE_BYTES]) before the first sw_append.  Every rank must
 * then make the same sw_append / sw_divide_rounds / ... calls. */
#define SW_PEER_HANDLE_BYTES 128
int sw_peer_handle(sw_engine *e, void *handle_out);
int sw_peer_connect(sw_engine *e, int rank, int nranks, const void *handles);

int sw_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SWIRLD_B200_H */
