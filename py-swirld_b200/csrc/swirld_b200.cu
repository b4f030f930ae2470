// swirld_b200.cu -- host side of libswirld_b200.so: the C ABI of include/swirld_b200.h
// over the kernels in swirld_*.cuh.  No torch, no CPU compute path: every
// consensus result is produced by a kernel; the host only validates the graph shape
// on append (what Node.is_valid_event checks, swirld.py:104-108), keeps the
// creator/height/chain-position mirrors it needs for that, and moves bytes.
#include "swirld_kernels.cuh"
#include "swirld_cansee.cuh"
#include "swirld_rounds.cuh"
#include "swirld_rcluster.cuh"
#include "swirld_wide.cuh"
#include "swirld_stream.cuh"
#include "swirld_verify.cuh"

#include <cstdlib>
#include "../../include/swirld_b200.h"

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <array>
#include <string>
#include <unordered_map>
#include <vector>

namespace {

std::string g_create_error;

// 32-byte event ids (BLAKE2b, swirld.py:95) -> arrival index
using Id32 = std::array<uint64_t, 4>;
struct Id32Hash { size_t operator()(const Id32 &k) const { return (size_t)(k[0] ^ (k[1] * 0x9E3779B97F4A7C15ull)); } };

struct TimedSpan { cudaEvent_t a, b; int cat; };

}  // namespace

struct sw_engine {
    int M = 0, NC = 1, cap = 0, C = 6, device = 0, Rcap = 0;
    int NJ = 1;                   // words per member set on the wide path: next power of two >= ceil(M/32)
    int MS = 64;                  // per-round array stride of find_order (64, or M on the wide path)
    int MP = 64;                  // max(M, 64): size of the per-member scratch arrays
    bool wide = false;            // swirld_wide.cuh kernels (M > 64, or SW_FORCE_WIDE=1)
    bool unit = true;
    i64 tot = 0;
    std::vector<i64> h_stake;
    // host mirrors for validation / views
    std::vector<int32_t> h_creator, h_head, h_count;
    int32_t *h_height = nullptr, *h_seq = nullptr;   // pinned, cap entries: sources of asynchronous copies
    uint8_t *h_stale = nullptr;                      // pinned: the other-parent is not its member's latest event
    cudaStream_t copy_stream = nullptr;              // sw_append's copies run beside the kernels of earlier chunks
    struct PendingAppend { int base; cudaEvent_t done; };
    std::vector<PendingAppend> appends;              // copies (+ eager can_see scans) the compute stream has not waited for yet
    cudaEvent_t scan_ev = nullptr;                   // last can_see scan issued on the compute stream
    bool scan_ev_set = false;
    int n_events = 0, n_divided = 0, n_tx = 0;
    // device columns
    int32_t *d_p0 = nullptr, *d_p1 = nullptr, *d_creator = nullptr, *d_seq = nullptr, *d_height = nullptr;
    uint8_t *d_stale = nullptr;
    long long *d_dbg = nullptr;
    unsigned rb_epoch = 0;        // launches of the round kernel (mask-cache key)
    int n_sm = 0;
    int32_t *d_Wf = nullptr, *d_cev = nullptr, *d_rbmeta = nullptr, *d_rbtot = nullptr, *d_gchain = nullptr;   // round-batch state
    ulonglong2 *d_sc = nullptr;
    uint8_t *d_res = nullptr;
    // cluster round kernel (swirld_rcluster.cuh): seq-space rows of the current chunk, hand-over state
    int32_t *d_rsg = nullptr, *d_rccont = nullptr;
    size_t rsg_cap = 0;           // events d_rsg holds
    bool rc_ok = false;           // a 16-CTA cluster with its shared memory can be resident on this device
    bool rc_mb = true;            // its exchanges by st.async + mbarrier (SW_RC_MB=0: plain stores + cluster barriers)
    int rc_min_n = 2048;          // shorter chunks go to the grid-wide kernel directly
    RcParams *d_rcviews = nullptr;
    RbParams *d_views = nullptr;  // sw_batch_divide_rounds: the views' parameters (owned by the first engine of a batch)
    int views_cap = 0;
    cudaEvent_t view_ev = nullptr;
    int n_rowed = 0;              // events whose can_see row is complete
    // can_see scan scratch (swirld_cansee.cuh)
    int4 *d_cs_meta = nullptr;
    uint8_t *d_cs_wr = nullptr, *d_cs_xb = nullptr, *d_cs_sflag = nullptr;
    int32_t *d_cs_last = nullptr, *d_cs_Q = nullptr, *d_cs_carry = nullptr, *d_cs_slow = nullptr, *d_cs_slowcnt = nullptr, *d_cs_xlist = nullptr, *d_cs_slowblk = nullptr, *d_cs_blkcnt = nullptr;
    std::vector<int32_t> h_stale_cum;    // h_stale_cum[i] = stale other-parents among events [0, i)
    int cs_min_B = 256;           // smallest block length the scan uses (sizes the per-block scratch)
    double *d_t = nullptr;
    uint8_t *d_sig = nullptr;
    int32_t *d_row = nullptr, *d_round = nullptr;
    u64 *d_SM = nullptr;
    uint8_t *d_wit = nullptr;
    int8_t *d_famous_ev = nullptr;
    // wide path
    unsigned *d_scw = nullptr, *d_SMw = nullptr, *d_Sw = nullptr;
    u64 *d_sctag = nullptr, *d_hitmin = nullptr;
    // several GPUs (sw_peer_connect): tests of a round step sharded by chain, first hits exchanged over NVLink
    int rank = 0, nranks = 1;
    void *d_xbuf = nullptr;       // [flags: 64 x u32][hits: 8 x 3 x M x u64], IPC-exported
    void *x_peer[8] = {nullptr};  // the same buffer of every rank (own: d_xbuf)
    int32_t *row_peer[8] = {nullptr};   // every rank's can_see table (own: d_row)
    unsigned **d_xflags2 = nullptr;     // device array of the ranks' barrier flag rows (xbuf + 128 bytes)
    unsigned xbar_count = 0;      // cross-GPU barriers issued so far (identical on every rank)
    unsigned *d_xstep = nullptr;  // steps published so far (device-resident: the step count of a launch is data dependent)
    // per round
    int32_t *d_W = nullptr, *d_rem = nullptr, *d_newc = nullptr;
    u64 *d_S = nullptr;
    int8_t *d_famous = nullptr;
    uint8_t *d_consensus = nullptr, *d_done = nullptr, *d_coin = nullptr;
    i64 *d_stake = nullptr;
    int32_t *d_scal = nullptr;
    // find_order
    int32_t *d_lastord = nullptr, *d_tx = nullptr, *d_idx = nullptr, *d_batch_ev = nullptr,
            *d_batch_seg = nullptr, *d_seg_start = nullptr, *d_seg_fw = nullptr, *d_seg_nf = nullptr,
            *d_perm = nullptr, *d_rounds_in = nullptr, *d_plan = nullptr;
    uint8_t *d_seg_white = nullptr;
    double *d_ts = nullptr;
    u64 *d_key = nullptr;
    int seg_cap = 0;
    void *d_flush = nullptr;
    size_t flush_bytes = 0;
    // small appends (the reference's cadence: one sync per call): one packed copy instead of eight
    static constexpr int STAGE_SLOTS = 8, STAGE_EVENTS = 64;
    uint8_t *h_stage = nullptr, *d_stage = nullptr;
    cudaEvent_t stage_ev[STAGE_SLOTS] = {nullptr};
    int stage_next = 0;
    int stream_n = 16;            // divide_rounds calls of at most this many events take the one-launch path (SW_STREAM_N)
    int32_t *h_scal = nullptr;    // pinned
    int32_t *h_newc = nullptr;    // pinned, Rcap
    cudaStream_t stream = nullptr;
    cudaEvent_t user_ev[16] = {nullptr};
    std::vector<TimedSpan> spans;
    std::vector<cudaEvent_t> pool;
    std::unordered_map<Id32, int32_t, Id32Hash> ids;     // sw_ingest: event id -> arrival index
    // signature / id checks (swirld_verify.cuh): member keys, their comb tables (+ B's), the inputs of the last check
    bool keys_set = false;
    uint8_t *d_vpk = nullptr, *d_vkeyok = nullptr;
    swv::Point *d_vbase = nullptr;
    swv::Precomp *d_vtab = nullptr;
    struct VBuf { void *p = nullptr; size_t cap = 0; };
    VBuf vbuf[9];
    int v_grid = 0;               // CTAs of k_verify that fit the device at once
    sw_stats_t stats{};
    std::string err;
};

namespace {

int fail(sw_engine *e, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (e) e->err = buf; else g_create_error = buf;
    return code;
}

#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t _s = (call);                                                         \
        if (_s != cudaSuccess)                                                           \
            return fail(e, SW_E_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(_s),   \
                        __FILE__, __LINE__);                                             \
    } while (0)

// call F<NJ>(args) for the engine's word count
#define SW_NJ(F, ...)                                                                    \
    (e->NJ == 1 ? F<1>(__VA_ARGS__) : e->NJ == 2 ? F<2>(__VA_ARGS__) : e->NJ == 4 ? F<4>(__VA_ARGS__) \
     : e->NJ == 8 ? F<8>(__VA_ARGS__) : e->NJ == 16 ? F<16>(__VA_ARGS__) : F<32>(__VA_ARGS__))

template <typename T>
cudaError_t dalloc(T **p, size_t n) { return cudaMalloc((void **)p, std::max<size_t>(n, 1) * sizeof(T)); }

cudaEvent_t get_event(sw_engine *e) {
    if (!e->pool.empty()) { cudaEvent_t ev = e->pool.back(); e->pool.pop_back(); return ev; }
    cudaEvent_t ev;
    cudaEventCreate(&ev);
    return ev;
}

struct Span {
    sw_engine *e; TimedSpan s;
    Span(sw_engine *e_, int cat) : e(e_) { s.a = get_event(e); s.b = get_event(e); s.cat = cat; cudaEventRecord(s.a, e->stream); }
    ~Span() { cudaEventRecord(s.b, e->stream); e->spans.push_back(s); }
};

void fold_spans(sw_engine *e) {
    std::vector<TimedSpan> pending;
    for (auto &s : e->spans) {
        if (cudaEventQuery(s.b) == cudaErrorNotReady) { pending.push_back(s); continue; }   // (a scan still running on the copy stream)
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) {
            if (s.cat == 0) e->stats.ms_divide_rounds += ms;
            else if (s.cat == 1) e->stats.ms_decide_fame += ms;
            else if (s.cat == 2) e->stats.ms_find_order += ms;
            else if (s.cat == 3) { e->stats.ms_can_see += ms; e->stats.ms_divide_rounds += ms; }
            else if (s.cat == 4) e->stats.ms_rounds_kernel += ms;
        }
        e->pool.push_back(s.a); e->pool.push_back(s.b);
    }
    e->spans.swap(pending);
}

// Make the compute stream wait for the appended batches that start below `upto` (all of them: upto < 0).
int wait_appends(sw_engine *e, int upto) {
    size_t k = 0;
    for (auto &a : e->appends) {
        if (upto >= 0 && a.base >= upto) { e->appends[k++] = a; continue; }
        CK(cudaStreamWaitEvent(e->stream, a.done, 0));
        e->pool.push_back(a.done);           // (re-recorded only after later work was enqueued behind the wait)
    }
    e->appends.resize(k);
    return 0;
}

int device_error(sw_engine *e) {     // after a sync: did a kernel flag an error?
    int code = e->h_scal[SC_ERR];
    if (code < 0) {
        const char *what = code == SW_E_CAPACITY ? "round table exhausted"
                         : code == SW_E_INDEX ? "list index out of range (swirld.py:305: a single seer)"
                         : code == SW_E_KEY ? "KeyError (undecided witness in a consensus round)"
                         : code == SW_E_CUDA ? "an exchange inside the round kernel timed out (a peer GPU, or a CTA of the cluster kernel, did not publish its step)" : "device error";
        return fail(e, code, "%s", what);
    }
    return 0;
}

int reset_state(sw_engine *e, bool keep_events = false) {
    const size_t RM = (size_t)e->Rcap * e->M;
    k_fill_i32<<<256, 256, 0, e->stream>>>(e->d_W, -1, RM);
    CK(cudaMemsetAsync(e->d_famous, 0xff, RM, e->stream));
    CK(cudaMemsetAsync(e->d_consensus, 0, e->Rcap, e->stream));
    CK(cudaMemsetAsync(e->d_famous_ev, 0xff, e->cap, e->stream));
    k_fill_i32<<<256, 256, 0, e->stream>>>(e->d_idx, -1, (size_t)e->cap);
    k_fill_i32<<<4, 256, 0, e->stream>>>(e->d_lastord, -1, (size_t)e->MP);
    k_fill_i32<<<4, 256, 0, e->stream>>>(e->d_cs_carry, -1, (size_t)e->MP);
    k_fill_i32<<<256, 256, 0, e->stream>>>(e->d_Wf, -1, RM);
    CK(cudaMemsetAsync(e->d_rbtot, 0, sizeof(int32_t) * e->MP, e->stream));
    k_fill_i32<<<64, 256, 0, e->stream>>>(e->d_gchain, -1, (size_t)e->MP * RB_RING);
    if (e->wide) {
        CK(cudaMemsetAsync(e->d_Sw, 0, RM * e->NJ * sizeof(unsigned), e->stream));
        CK(cudaMemsetAsync(e->d_sctag, 0, sizeof(u64) * (size_t)e->cap, e->stream));
    } else {
        CK(cudaMemsetAsync(e->d_S, 0, RM * sizeof(u64), e->stream));
        CK(cudaMemsetAsync(e->d_sc, 0, sizeof(ulonglong2) * (size_t)e->cap, e->stream));
    }
    int32_t sc[SC_COUNT] = {0};
    sc[SC_MAX_ROUND] = -1;
    CK(cudaMemcpyAsync(e->d_scal, sc, sizeof sc, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->stats.kernel_launches += 5;
    e->n_divided = e->n_tx = 0;
    e->n_rowed = 0;
    e->rb_epoch = 0;
    if (!keep_events) {
        e->n_events = 0;
        std::fill(e->h_head.begin(), e->h_head.end(), -1);
        std::fill(e->h_count.begin(), e->h_count.end(), 0);
    }
    memset(e->h_scal, 0, sizeof(int32_t) * SC_COUNT);
    return 0;
}

// can_see rows of the appended events [n_rowed, upto): the column-tiled blocked scan of swirld_cansee.cuh.
// `st`: the compute stream (lazily, from sw_divide_rounds) or the copy stream (eagerly, from sw_append: the
// scan of a new chunk then runs beside the round kernel of the previous one).  The two never overlap: a scan
// on one stream first waits for the last scan issued on the other (they share the scratch and the carry heads).
int cansee_scan(sw_engine *e, cudaStream_t st, int upto) {
    const int first = e->n_rowed, n = upto - e->n_rowed;
    if (n <= 0) return 0;
    const int M = e->M;
    CsParams C{};
    C.M = M; C.first = first; C.n = n;
    C.p0 = e->d_p0; C.p1 = e->d_p1; C.creator = e->d_creator; C.stale = e->d_stale; C.row = e->d_row;
    C.meta = e->d_cs_meta; C.wr = e->d_cs_wr; C.xb = e->d_cs_xb; C.last = e->d_cs_last; C.Qtab = e->d_cs_Q;
    C.carry = e->d_cs_carry; C.slow_list = e->d_cs_slow; C.slow_cnt = e->d_cs_slowcnt; C.sflag = e->d_cs_sflag; C.xlist = e->d_cs_xlist; C.slow_blk = e->d_cs_slowblk; C.blk_cnt = e->d_cs_blkcnt;
    cudaEvent_t a = get_event(e), b = get_event(e);
    int small_n = 24;
    if (const char *v = getenv("SW_CS_SMALL")) small_n = atoi(v);
    if (n <= small_n) {                                // the reference's own cadence: a handful of events per call
        cudaEventRecord(a, st);
        k_cs_small<<<1, std::min(1024, (M + 31) / 32 * 32), 0, st>>>(C);
        cudaEventRecord(b, st);
        e->spans.push_back(TimedSpan{a, b, 3});
        CK(cudaGetLastError());
        e->stats.kernel_launches += 1;
        e->n_rowed = upto;
        return 0;
    }
    // block length: >= 16 (32 above 64 members) events per member and block, so that nearly every member's last event of a
    // block sees every block-start head (then the finality check passes; the rest goes through the waves); SW_CS_B overrides
    int B = std::max(e->cs_min_B, std::min((M <= 64 ? 16 : 32) * M, 1 << 15));      // (above 64 members seeing every head takes more events per member)
    if (const char *v = getenv("SW_CS_B")) B = std::max(e->cs_min_B, atoi(v));
    B = (B + 3) & ~3;
    C.B = B;
    C.first_al = first & ~3;
    C.nb = (first + n <= C.first_al + B) ? 1 : 1 + (first + n - (C.first_al + B) + B - 1) / B;
    if (C.nb > 1 && first + n - (C.first_al + (C.nb - 1) * B) < 3 * B / 4) C.nb--;     // a short tail joins the block before it
    // columns per tile: 32 (one warp = one 128-byte row segment) unless the per-member cache val[M][CT] then limits a
    // SM to so few CTAs that narrower tiles finish in fewer waves (M = 1024: 128 KB per CTA at CT = 32)
    const bool has_stale = e->h_stale_cum[first + n] - e->h_stale_cum[first] > 0;
    C.SV = has_stale ? CS_SV : 0;
    int CT = 32;
    {
        long long best = -1;
        for (int ct = 32; ct >= 8; ct >>= 1) {
            const long long smem_ct = (long long)(M + C.SV) * ct * 4 + CS_TILE * 16 + 3 * CS_TILE;
            const long long conc = std::max(1LL, std::min(32LL, (220LL << 10) / smem_ct));
            const long long ctas = (long long)C.nb * ((M + ct - 1) / ct);
            const long long waves = (ctas + e->n_sm * conc - 1) / (e->n_sm * conc);
            if (best < 0 || waves < best) { best = waves; CT = ct; }
        }
    }
    if (const char *v = getenv("SW_CS_CT")) { const int x = atoi(v); if (x == 8 || x == 16 || x == 32) CT = x; }
    C.CT = CT;
    int tile_lo = 0, tile_hi = (M + CT - 1) / CT;
    bool shard = e->nranks > 1;
    if (const char *v = getenv("SW_CS_SHARD")) shard = shard && atoi(v) != 0;       // (0: every rank computes the whole table itself)
    if (shard) {                                          // the column tiles of this rank; every rank stores into every table
        const int nt = tile_hi;
        tile_lo = (int)((long long)nt * e->rank / e->nranks); tile_hi = (int)((long long)nt * (e->rank + 1) / e->nranks);
        C.npeer = e->nranks;
        for (int p = 0; p < e->nranks; p++) C.prow[p] = e->row_peer[p];
    }
    C.tile_lo = tile_lo;
    const int ntiles = std::max(0, tile_hi - tile_lo);
    auto xbarrier = [&]() -> int {
        if (!shard) return 0;
        k_xbarrier<<<1, 32, 0, st>>>(e->d_xflags2, e->rank, e->nranks, ++e->xbar_count, e->d_scal);
        CK(cudaGetLastError());
        return 0;
    };
    const size_t smem = (size_t)(M + C.SV) * CT * sizeof(int) + CS_TILE * sizeof(int4) + 3 * CS_TILE;
    const int pblocks = std::max(1, std::min(8 * e->n_sm, (n + 255) / 256));
    k_fill_i32<<<std::max(1, std::min(256, (int)(((size_t)C.nb * M + 255) / 256))), 256, 0, st>>>(e->d_cs_last, -1, (size_t)C.nb * M);
    if (C.nb > 1) {
        CK(cudaMemsetAsync(e->d_cs_wr + first, 0, (size_t)n, st));
        CK(cudaMemsetAsync(e->d_cs_xb + (first & ~3), 0, (size_t)(n + (first & 3)), st));
        CK(cudaMemsetAsync(e->d_cs_sflag + first, 0, (size_t)n, st));
        CK(cudaMemsetAsync(e->d_cs_slowcnt, 0, sizeof(int32_t) * 4, st));
        CK(cudaMemsetAsync(e->d_cs_blkcnt, 0, sizeof(int32_t) * (size_t)C.nb, st));
    }
    cudaEventRecord(a, st);
    k_cs_prep<<<pblocks, 256, 0, st>>>(C);
    if (C.nb > 1) {
        if (ntiles > 0) {
            const dim3 g(C.nb, ntiles);
            if (shard) { if (has_stale) k_cs_pass<1, true, true><<<g, CS_CT, smem, st>>>(C); else k_cs_pass<1, false, true><<<g, CS_CT, smem, st>>>(C); }
            else { if (has_stale) k_cs_pass<1, true, false><<<g, CS_CT, smem, st>>>(C); else k_cs_pass<1, false, false><<<g, CS_CT, smem, st>>>(C); }
        }
        if (xbarrier() < 0) return SW_E_CUDA;              // every rank's partial rows are in every table
    }
    k_cs_heads<<<std::max(1, std::min(2 * e->n_sm, (int)(((size_t)(C.nb + 1) * M + 255) / 256))), 256, 0, st>>>(C);
    if (C.nb > 1) {
        k_cs_check<<<std::max(1, std::min(4 * e->n_sm, (int)(((size_t)C.nb * M + 7) / 8))), 256, 0, st>>>(C);
        const size_t ssm = (size_t)CS_SLOW_WARPS * M * sizeof(int);
        k_cs_slow_wave<<<e->n_sm, CS_SLOW_WARPS * 32, ssm, st>>>(C, 1);
        k_cs_slow_wave<<<e->n_sm, CS_SLOW_WARPS * 32, ssm, st>>>(C, 2);
        k_cs_slow_rest<<<1, CS_REST_WARPS * 32, (size_t)CS_REST_WARPS * M * sizeof(int), st>>>(C);
    }
    if (ntiles > 0) {
        const dim3 g(C.nb, ntiles);
        if (shard) { if (has_stale) k_cs_pass<2, true, true><<<g, CS_CT, smem, st>>>(C); else k_cs_pass<2, false, true><<<g, CS_CT, smem, st>>>(C); }
        else { if (has_stale) k_cs_pass<2, true, false><<<g, CS_CT, smem, st>>>(C); else k_cs_pass<2, false, false><<<g, CS_CT, smem, st>>>(C); }
    }
    if (shard) k_cs_carry<<<(M + 255) / 256, 256, 0, st>>>(C);
    if (xbarrier() < 0) return SW_E_CUDA;                  // the whole table is in every rank's memory
    cudaEventRecord(b, st);
    e->spans.push_back(TimedSpan{a, b, 3});
    CK(cudaGetLastError());
    e->stats.kernel_launches += C.nb > 1 ? 9 : 4;
    e->n_rowed = upto;
    return 0;
}

// rounds of the chunk by the cooperative round-batch kernel (swirld_rounds.cuh), M <= 64: parameters + the kernels
// that group the chunk's events by creator (`grid` = CTAs this view's round kernel will run on)
int round_batch_prep(sw_engine *e, int first, int n, int grid, RbParams &R, int min_L = 1) {
    R = RbParams{};
    R.M = e->M; R.first = first; R.n = n; R.Rcap = e->Rcap;
    R.L = std::max(std::min(min_L, RB_LMAX), std::min(RB_LMAX, grid * (RB_THREADS / 32) / e->M));
    R.maxmiss = RB_MAXMISS;
    R.epoch = ++e->rb_epoch;
    if (const char *v = getenv("SW_RB_L")) R.L = std::max(1, std::min(R.L, atoi(v)));          // tuning knobs
    if (const char *v = getenv("SW_RB_MAXMISS")) R.maxmiss = std::max(0, atoi(v));
    R.row = e->d_row; R.p0 = e->d_p0; R.creator = e->d_creator; R.seq = e->d_seq; R.round = e->d_round;
    R.Wf = e->d_Wf; R.sc = e->d_sc; R.cev = e->d_cev;
    R.ccnt = e->d_rbmeta; R.cmin = e->d_rbmeta + 64; R.coff = e->d_rbmeta + 128; R.bar = reinterpret_cast<unsigned *>(e->d_rbmeta + 224);
    R.ctot = e->d_rbtot; R.gchain = e->d_gchain;
    R.res = e->d_res; R.stake = e->d_stake; R.tot2 = 2 * e->tot; R.scal = e->d_scal;
    R.wit = e->d_wit; R.W = e->d_W; R.SM = e->d_SM; R.dbg = e->d_dbg;
    R.wlist = e->d_cev + e->cap; R.wcnt = e->d_rbmeta + 225;
    CK(cudaMemsetAsync(R.ccnt, 0, sizeof(int32_t) * 64, e->stream));
    CK(cudaMemsetAsync(R.cmin, 0x7f, sizeof(int32_t) * 64, e->stream));
    const int blocks = std::max(1, std::min(296, (n + 255) / 256));
    k_rb_count<<<blocks, 256, 0, e->stream>>>(R);
    k_rb_offsets<<<1, 32, 0, e->stream>>>(R);
    k_rb_scatter<<<blocks, 256, 0, e->stream>>>(R);
    CK(cudaGetLastError());
    return 0;
}

// what follows the round kernel: ring of recent events, witness flags / table / list, seen-masks, strongly-seen sets
template <int NC>
int round_batch_finish(sw_engine *e, const RbParams &R) {
    const int n = R.n, blocks = std::max(1, std::min(296, (n + 255) / 256));
    k_rb_tail<<<blocks, 256, 0, e->stream>>>(R);
    k_rb_witness<<<blocks, 256, 0, e->stream>>>(R);
    k_rb_seenmask<NC><<<(n + 7) / 8, 256, 0, e->stream>>>(R);
    CK(cudaGetLastError());
    StrongParams Q{};
    Q.M = e->M; Q.first = R.first; Q.n = n; Q.Rcap = e->Rcap; Q.creator = e->d_creator; Q.row = e->d_row;
    Q.round = e->d_round; Q.wit = e->d_wit; Q.SM = e->d_SM; Q.S = e->d_S; Q.stake = e->d_stake; Q.tot2 = 2 * e->tot;
    Q.coin = e->d_coin; Q.sig = e->d_sig; Q.unit = e->unit ? 1 : 0;
    Q.list = R.wlist; Q.list_n = R.wcnt;
    const int sblocks = std::max(1, std::min((n + 7) / 8, 4 * e->n_sm));
    k_strong<NC><<<sblocks, 256, 0, e->stream>>>(Q);
    CK(cudaGetLastError());
    e->stats.kernel_launches += 8;
    return 0;
}

// seq-space rows of the chunk for the cluster round kernel (after round_batch_prep grouped the chunk by creator)
int rc_seqrows(sw_engine *e, const RbParams &R) {
    const int n = R.n;
    if ((size_t)n > e->rsg_cap) {
        if (e->d_rsg) { CK(cudaStreamSynchronize(e->stream)); CK(cudaFree(e->d_rsg)); e->d_rsg = nullptr; e->rsg_cap = 0; }
        const size_t want = std::min<size_t>((size_t)e->cap, std::max<size_t>((size_t)n, 1 << 16));
        CK(dalloc(&e->d_rsg, want * 64));
        e->rsg_cap = want;
    }
    k_rc_seqrows<<<std::max(1, std::min(4 * e->n_sm, (n + 7) / 8)), 256, 0, e->stream>>>(R, e->d_rsg);
    CK(cudaGetLastError());
    return 0;
}
void rc_launch_config(cudaLaunchConfig_t &cfg, cudaLaunchAttribute *at, int clusters, cudaStream_t stream) {
    cfg = cudaLaunchConfig_t{};
    cfg.gridDim = dim3(RC_CS * clusters); cfg.blockDim = dim3(RC_THREADS); cfg.dynamicSmemBytes = RC_SMEM_BYTES; cfg.stream = stream;
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = RC_CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
}

template <int NC, bool UNIT>
int divide_round_batch(sw_engine *e, int first, int n) {
    // a few SMs stay free for the can_see scan of the next chunk, which runs beside this kernel (SW_RB_FREE_SMS)
    int free_sms = 16;
    if (const char *v = getenv("SW_RB_FREE_SMS")) free_sms = std::max(0, atoi(v));
    const int grid = std::max(e->n_sm / 2, e->n_sm - free_sms);
    RbParams R;
    if (round_batch_prep(e, first, n, grid, R) < 0) return SW_E_CUDA;
    void *args[] = {(void *)&R};
    {
        cudaEvent_t a = get_event(e), b = get_event(e);
        cudaEventRecord(a, e->stream);
        if (e->rc_ok && n >= e->rc_min_n) {
            // the chunk inside one thread-block cluster; k_rounds_batch takes over whatever it hands back (normally nothing)
            if (rc_seqrows(e, R) < 0) return SW_E_CUDA;
            RcParams Q{R, e->d_rsg, e->d_rccont};
            cudaLaunchConfig_t cfg;
            cudaLaunchAttribute at[1];
            rc_launch_config(cfg, at, 1, e->stream);
            if (e->rc_mb) CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster<UNIT, true>, Q));
            else CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster<UNIT, false>, Q));
            R.cont = e->d_rccont;
            e->stats.kernel_launches += 2;
        }
        CK(cudaLaunchCooperativeKernel((void *)k_rounds_batch<NC, UNIT>, dim3(grid), dim3(RB_THREADS), args, 0, e->stream));
        cudaEventRecord(b, e->stream);
        e->spans.push_back(TimedSpan{a, b, 4});
    }
    return round_batch_finish<NC>(e, R);
}

size_t rounds_wide_smem(int M) { return (size_t)(2 * M + 16 * M + 1 + 32 + (RW_THREADS / 32) * M + 1) * sizeof(int); }

// rounds of the chunk for any member count (swirld_wide.cuh)
template <int NJ>
int divide_rounds_wide(sw_engine *e, int first, int n) {
    const int M = e->M;
    RwParams R{};
    R.M = M; R.first = first; R.n = n; R.Rcap = e->Rcap;
    const int grid = e->n_sm;
    const int nw = grid * (RW_THREADS / 32);
    const int nown = (M + e->nranks - 1) / e->nranks;
    // events per member below a step's frontier: about three tests per warp and step, never more than half a window
    R.L = std::max(1, std::min(RW_LMAX / 2, 3 * nw * e->nranks / std::max(1, M)));
    (void)nown;
    if (const char *v = getenv("SW_RW_L")) R.L = std::max(1, std::min(RW_LMAX, atoi(v)));
    R.epoch = ++e->rb_epoch;
    R.row = e->d_row; R.p0 = e->d_p0; R.creator = e->d_creator; R.seq = e->d_seq; R.round = e->d_round;
    R.Wf = e->d_Wf; R.scw = e->d_scw; R.sctag = e->d_sctag; R.cev = e->d_cev;
    R.ccnt = e->d_rbmeta; R.cmin = e->d_rbmeta + M; R.coff = e->d_rbmeta + 2 * M; R.bar = reinterpret_cast<unsigned *>(e->d_rbmeta + 3 * M + 8);
    int32_t *wcnt = e->d_rbmeta + 3 * M + 9, *wlist = e->d_cev + e->cap;
    R.ctot = e->d_rbtot; R.gchain = e->d_gchain; R.hitmin = e->d_hitmin; R.ticket = reinterpret_cast<unsigned *>(e->d_rbmeta + 3 * M + 12);
    R.stake = e->d_stake; R.tot2 = 2 * e->tot; R.unit = e->unit ? 1 : 0; R.scal = e->d_scal; R.dbg = e->d_dbg;
    R.rank = e->rank; R.nranks = e->nranks; R.xstep = e->d_xstep;
    for (int p = 0; p < e->nranks && p < 8; p++) {
        R.xflag[p] = reinterpret_cast<unsigned *>(e->x_peer[p]);
        R.xhit[p] = reinterpret_cast<u64 *>(reinterpret_cast<char *>(e->x_peer[p]) + 256);
    }
    CK(cudaMemsetAsync(R.ccnt, 0, sizeof(int32_t) * M, e->stream));
    CK(cudaMemsetAsync(R.cmin, 0x7f, sizeof(int32_t) * M, e->stream));
    const int blocks = std::max(1, std::min(2 * e->n_sm, (n + 255) / 256));
    k_rw_count<<<blocks, 256, 0, e->stream>>>(R);
    k_rw_offsets<<<1, 1024, 0, e->stream>>>(R, wcnt);
    k_rw_scatter<<<blocks, 256, 0, e->stream>>>(R);
    CK(cudaGetLastError());
    const size_t smem = rounds_wide_smem(M);
    CK(cudaFuncSetAttribute(k_rounds_wide<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    void *args[] = {(void *)&R};
    {
        cudaEvent_t a = get_event(e), b = get_event(e);
        cudaEventRecord(a, e->stream);
        CK(cudaLaunchCooperativeKernel((void *)k_rounds_wide<NJ>, dim3(grid), dim3(RW_THREADS), args, smem, e->stream));
        cudaEventRecord(b, e->stream);
        e->spans.push_back(TimedSpan{a, b, 4});
    }
    RbParams T{};                                      // the finish kernels shared with the M <= 64 path
    T.M = M; T.first = first; T.n = n; T.Rcap = e->Rcap; T.p0 = e->d_p0; T.creator = e->d_creator; T.seq = e->d_seq;
    T.round = e->d_round; T.ctot = e->d_rbtot; T.gchain = e->d_gchain; T.wit = e->d_wit; T.W = e->d_W;
    T.wlist = wlist; T.wcnt = wcnt;
    k_rb_tail<<<blocks, 256, 0, e->stream>>>(T);
    k_rb_witness<<<blocks, 256, 0, e->stream>>>(T);
    k_w_seenmask<NJ><<<std::max(1, std::min(8 * e->n_sm, (n + 7) / 8)), 256, 0, e->stream>>>(M, first, n, e->Rcap, e->d_row, e->d_round, e->d_W, e->d_SMw);
    CK(cudaGetLastError());
    StrongParams Q{};
    Q.M = M; Q.first = first; Q.n = n; Q.Rcap = e->Rcap; Q.creator = e->d_creator; Q.row = e->d_row;
    Q.round = e->d_round; Q.wit = e->d_wit; Q.stake = e->d_stake; Q.tot2 = 2 * e->tot;
    Q.coin = e->d_coin; Q.sig = e->d_sig; Q.unit = e->unit ? 1 : 0; Q.list = wlist; Q.list_n = wcnt;
    Q.SMw = e->d_SMw; Q.Sw = e->d_Sw;
    const size_t ssm = (size_t)(2 * M + 8 * M) * sizeof(int);
    CK(cudaFuncSetAttribute(k_w_strong<NJ>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ssm));
    k_w_strong<NJ><<<std::max(1, std::min(4 * e->n_sm, (n + 7) / 8)), 256, ssm, e->stream>>>(Q);
    CK(cudaGetLastError());
    e->stats.kernel_launches += 8;
    return 0;
}

template <int NJ>
int fame_rounds_wide(sw_engine *e, const FameParams &P) {
    const size_t smem = (size_t)(32 * NJ + 64) * sizeof(int) + (size_t)(32 + e->M) * sizeof(i64);
    const int parts = (e->M + FW_THREADS - 1) / FW_THREADS;
    k_w_fame_rounds<NJ><<<(2 * e->n_sm / parts + 1) * parts, FW_THREADS, smem, e->stream>>>(P);
    return 0;
}

}  // namespace

extern "C" {

int sw_version(void) { return 200; }

const char *sw_last_error(const sw_engine *e) { return e ? e->err.c_str() : g_create_error.c_str(); }

int sw_create(int M, int capacity_events, const int64_t *stake, int coin_period, int device,
              sw_engine **out) {
    sw_engine *e = nullptr;
    if (!out) return fail(e, SW_E_ARG, "out is NULL");
    *out = nullptr;
    if (M < 1 || capacity_events < 1 || coin_period < 1) return fail(e, SW_E_ARG, "bad M / capacity / coin period");
    if (M > SW_MAX_MEMBERS) return fail(e, SW_E_UNSUPPORTED, "M=%d > %d members not supported by this build", M, SW_MAX_MEMBERS);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(e, SW_E_CUDA, "no CUDA device (this engine has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(e, SW_E_ARG, "device %d out of range (%d devices)", device, ndev);
    e = new sw_engine();
    e->M = M; e->NC = (M + 31) / 32; e->cap = capacity_events; e->C = coin_period; e->device = device;
    e->wide = M > 64;
    if (const char *v = getenv("SW_FORCE_WIDE")) if (atoi(v)) e->wide = true;
    e->NJ = 1;
    while (e->NJ * 32 < M) e->NJ *= 2;
    e->MS = e->wide ? M : 64;
    e->MP = std::max(M, 64);
    e->h_stake.resize(M);
    for (int c = 0; c < M; c++) {
        e->h_stake[c] = stake ? stake[c] : 1;
        if (e->h_stake[c] < 0) { delete e; return fail(nullptr, SW_E_ARG, "negative stake"); }
        if (e->h_stake[c] != 1) e->unit = false;
        e->tot += e->h_stake[c];
    }
    // a round other than the last needs more than 2*tot/3 members with a witness (quirk Q3)
    i64 per = std::min<i64>(M, (2 * e->tot) / 3 + 1);
    if (per < 1) per = 1;
    e->Rcap = (int)std::min<i64>((i64)e->cap + 2, (i64)e->cap / per + 16);
    e->h_head.assign(M, -1);
    e->h_count.assign(M, 0);
    e->h_creator.reserve(e->cap);
    e->h_stale_cum.assign(1, 0);
    int rc = [&]() -> int {
        CK(cudaSetDevice(device));
        CK(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&e->scan_ev, cudaEventDisableTiming));
        const size_t cap = e->cap, RM = (size_t)e->Rcap * M, MP = e->MP;
        CK(cudaMallocHost((void **)&e->h_height, sizeof(int32_t) * cap));
        CK(cudaMallocHost((void **)&e->h_seq, sizeof(int32_t) * cap));
        CK(cudaMallocHost((void **)&e->h_stale, cap));
        CK(dalloc(&e->d_p0, cap)); CK(dalloc(&e->d_p1, cap)); CK(dalloc(&e->d_creator, cap)); CK(dalloc(&e->d_seq, cap));
        CK(dalloc(&e->d_t, cap)); CK(dalloc(&e->d_sig, cap * 64)); CK(dalloc(&e->d_height, cap)); CK(dalloc(&e->d_stale, cap));
        // can_see scan scratch: per-event meta / flags / slow list, per-block tables (blocks are >= cs_min_B events)
        e->cs_min_B = std::max(256, std::min((M <= 64 ? 16 : 32) * M, 1 << 15));
        if (const char *v = getenv("SW_CS_B")) e->cs_min_B = std::max(64, std::min(e->cs_min_B, atoi(v)));
        const size_t nbmax = cap / e->cs_min_B + 3;
        CK(dalloc(&e->d_cs_meta, cap)); CK(dalloc(&e->d_cs_wr, cap)); CK(dalloc(&e->d_cs_xb, cap)); CK(dalloc(&e->d_cs_slow, cap + 4));
        CK(dalloc(&e->d_cs_last, nbmax * M)); CK(dalloc(&e->d_cs_Q, (nbmax + 1) * M)); CK(dalloc(&e->d_cs_slowcnt, (size_t)4)); CK(dalloc(&e->d_cs_sflag, cap)); CK(dalloc(&e->d_cs_xlist, cap + 4)); CK(dalloc(&e->d_cs_slowblk, cap + 4)); CK(dalloc(&e->d_cs_blkcnt, nbmax + 1));
        CK(dalloc(&e->d_cs_carry, MP));
        CK(dalloc(&e->d_Wf, RM)); CK(dalloc(&e->d_cev, 2 * cap)); /* + the witness list of the current chunk */
        CK(dalloc(&e->d_rbmeta, std::max<size_t>(256, 3 * MP + 64)));
        CK(dalloc(&e->d_rbtot, MP)); CK(dalloc(&e->d_gchain, MP * RB_RING));
        CK(cudaDeviceGetAttribute(&e->n_sm, cudaDevAttrMultiProcessorCount, device));
        CK(dalloc(&e->d_dbg, (size_t)40)); CK(cudaMemsetAsync(e->d_dbg, 0, sizeof(long long) * 40, e->stream));
        CK(dalloc(&e->d_row, cap * M));
        if (e->wide) {
            CK(dalloc(&e->d_scw, cap * e->NJ)); CK(dalloc(&e->d_sctag, cap)); CK(dalloc(&e->d_SMw, cap * e->NJ));
            CK(dalloc(&e->d_Sw, RM * e->NJ)); CK(dalloc(&e->d_hitmin, (size_t)3 * M));
            CK(cudaMalloc(&e->d_xbuf, 256 + (size_t)8 * 3 * M * sizeof(u64)));
            CK(cudaMemsetAsync(e->d_xbuf, 0, 256 + (size_t)8 * 3 * M * sizeof(u64), e->stream));
            CK(dalloc(&e->d_xstep, (size_t)1)); CK(cudaMemsetAsync(e->d_xstep, 0, sizeof(unsigned), e->stream));
            e->x_peer[0] = e->d_xbuf;
        } else {
            CK(dalloc(&e->d_sc, cap)); CK(dalloc(&e->d_res, (size_t)2 * 64 * RB_LMAX));
            CK(dalloc(&e->d_SM, cap)); CK(dalloc(&e->d_S, RM));
            // the cluster round kernel: 16 CTAs with ~174 KB of shared memory each must fit one GPC
            CK(dalloc(&e->d_rccont, (size_t)132)); CK(cudaMemsetAsync(e->d_rccont, 0, sizeof(int32_t) * 132, e->stream));
            bool want = true;
            if (const char *v = getenv("SW_ROUNDS_CLUSTER")) want = atoi(v) != 0;
            if (const char *v = getenv("SW_RC_MIN_N")) e->rc_min_n = std::max(1, atoi(v));
            if (want) {
                int ncl = 0;
                if (const char *v = getenv("SW_RC_MB")) e->rc_mb = atoi(v) != 0;
                const void *fn = e->unit ? (e->rc_mb ? (const void *)k_rounds_cluster<true, true> : (const void *)k_rounds_cluster<true, false>)
                                         : (e->rc_mb ? (const void *)k_rounds_cluster<false, true> : (const void *)k_rounds_cluster<false, false>);
                cudaError_t er = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RC_SMEM_BYTES);
                if (er == cudaSuccess) er = cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
                if (er == cudaSuccess) {
                    const void *fv = e->unit ? (e->rc_mb ? (const void *)k_rounds_cluster_views<true, true> : (const void *)k_rounds_cluster_views<true, false>)
                                             : (e->rc_mb ? (const void *)k_rounds_cluster_views<false, true> : (const void *)k_rounds_cluster_views<false, false>);
                    er = cudaFuncSetAttribute(fv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RC_SMEM_BYTES);
                    if (er == cudaSuccess) er = cudaFuncSetAttribute(fv, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
                    cudaLaunchConfig_t cfg;
                    cudaLaunchAttribute at[1];
                    rc_launch_config(cfg, at, 1, nullptr);
                    if (er == cudaSuccess) er = cudaOccupancyMaxActiveClusters(&ncl, fv, &cfg);
                }
                e->rc_ok = er == cudaSuccess && ncl >= 1;
                if (er != cudaSuccess) (void)cudaGetLastError();
                if (getenv("SW_DEBUG")) fprintf(stderr, "swirld_b200: cluster round kernel %s (%s, %d clusters of %d CTAs resident)\n", e->rc_ok ? "on" : "off", cudaGetErrorString(er), ncl, RC_CS);
            }
        }
        CK(dalloc(&e->d_round, cap)); CK(dalloc(&e->d_wit, cap)); CK(dalloc(&e->d_famous_ev, cap));
        CK(dalloc(&e->d_W, RM)); CK(dalloc(&e->d_famous, RM));
        CK(dalloc(&e->d_consensus, (size_t)e->Rcap)); CK(dalloc(&e->d_done, (size_t)e->Rcap)); CK(dalloc(&e->d_coin, RM));
        CK(dalloc(&e->d_rem, (size_t)e->Rcap)); CK(dalloc(&e->d_newc, (size_t)e->Rcap));
        CK(dalloc(&e->d_stake, (size_t)M)); CK(dalloc(&e->d_scal, (size_t)SC_COUNT));
        CK(dalloc(&e->d_lastord, MP)); CK(dalloc(&e->d_tx, cap)); CK(dalloc(&e->d_idx, cap));
        CK(dalloc(&e->d_batch_ev, cap)); CK(dalloc(&e->d_batch_seg, cap)); CK(dalloc(&e->d_perm, 2 * cap));
        CK(dalloc(&e->d_ts, cap)); CK(dalloc(&e->d_key, cap * 8));
        const size_t slot = (unpack_bytes(sw_engine::STAGE_EVENTS) + 255) & ~(size_t)255;
        CK(cudaMallocHost((void **)&e->h_stage, slot * sw_engine::STAGE_SLOTS));
        CK(cudaMalloc((void **)&e->d_stage, slot * sw_engine::STAGE_SLOTS));
        for (auto &ev : e->stage_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        if (const char *v = getenv("SW_STREAM_N")) e->stream_n = std::max(0, std::min(1024, atoi(v)));
        CK(cudaFuncSetAttribute(k_stream_divide<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * 1024));
        CK(cudaMallocHost((void **)&e->h_scal, sizeof(int32_t) * SC_COUNT));
        CK(cudaMallocHost((void **)&e->h_newc, sizeof(int32_t) * e->Rcap));
        CK(cudaMemcpyAsync(e->d_stake, e->h_stake.data(), sizeof(i64) * M, cudaMemcpyHostToDevice, e->stream));
        // kernels that need more than the default 48 KB of dynamic shared memory
        const size_t cs_smem = (size_t)(M + CS_SV) * CS_CT * sizeof(int) + CS_TILE * sizeof(int4) + 3 * CS_TILE;
        CK(cudaFuncSetAttribute(k_cs_pass<1, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<1, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<2, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<1, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<2, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_pass<2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cs_smem));
        CK(cudaFuncSetAttribute(k_cs_slow_wave, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)CS_SLOW_WARPS * M * sizeof(int))));
        CK(cudaFuncSetAttribute(k_cs_slow_rest, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)CS_REST_WARPS * M * sizeof(int))));
        return reset_state(e);
    }();
    if (rc < 0) { g_create_error = e->err; sw_destroy(e); return rc; }
    memset(&e->stats, 0, sizeof e->stats);
    *out = e;
    return SW_OK;
}

void sw_destroy(sw_engine *e) {
    if (!e) return;
    cudaSetDevice(e->device);
    if (e->stream) { wait_appends(e, -1); cudaStreamSynchronize(e->stream); }
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    fold_spans(e);
    for (auto ev : e->pool) cudaEventDestroy(ev);
    for (auto ev : e->user_ev) if (ev) cudaEventDestroy(ev);
    if (e->scan_ev) cudaEventDestroy(e->scan_ev);
    if (e->view_ev) cudaEventDestroy(e->view_ev);
    if (e->d_views) cudaFree(e->d_views);
    if (e->d_rcviews) cudaFree(e->d_rcviews);
    for (auto ev : e->stage_ev) if (ev) cudaEventDestroy(ev);
    if (e->h_stage) cudaFreeHost(e->h_stage);
    if (e->d_stage) cudaFree(e->d_stage);
    for (int p = 0; p < 8; p++) if (e->x_peer[p] && e->x_peer[p] != e->d_xbuf) cudaIpcCloseMemHandle(e->x_peer[p]);
    for (int p = 0; p < 8; p++) if (e->row_peer[p] && e->row_peer[p] != e->d_row) cudaIpcCloseMemHandle(e->row_peer[p]);
    if (e->d_xflags2) cudaFree(e->d_xflags2);
    void *ptrs[] = {e->d_rbtot, e->d_gchain, e->d_Wf, e->d_cev, e->d_rbmeta, e->d_sc, e->d_res, e->d_cs_last, e->d_cs_Q, e->d_cs_carry,
                    e->d_cs_meta, e->d_cs_wr, e->d_cs_xb, e->d_cs_sflag, e->d_cs_xlist, e->d_cs_slowblk, e->d_cs_blkcnt, e->d_cs_slow, e->d_cs_slowcnt, e->d_stale, e->d_coin, e->d_dbg, e->d_height,
                    e->d_p0, e->d_p1, e->d_creator, e->d_seq, e->d_t, e->d_sig, e->d_row, e->d_SM,
                    e->d_scw, e->d_sctag, e->d_SMw, e->d_Sw, e->d_hitmin, e->d_xbuf, e->d_xstep,
                    e->d_round, e->d_wit, e->d_famous_ev, e->d_W, e->d_S, e->d_famous, e->d_consensus,
                    e->d_done, e->d_rem, e->d_newc, e->d_stake, e->d_scal, e->d_lastord, e->d_tx, e->d_idx,
                    e->d_batch_ev, e->d_batch_seg, e->d_perm, e->d_ts, e->d_key, e->d_seg_start, e->d_seg_fw,
                    e->d_seg_nf, e->d_seg_white, e->d_rounds_in, e->d_plan, e->d_flush, e->d_rsg, e->d_rccont};
    for (void *p : ptrs) if (p) cudaFree(p);
    void *vptrs[] = {e->d_vpk, e->d_vkeyok, e->d_vbase, e->d_vtab};
    for (void *p : vptrs) if (p) cudaFree(p);
    for (auto &b : e->vbuf) if (b.p) cudaFree(b.p);
    if (e->h_scal) cudaFreeHost(e->h_scal);
    if (e->h_newc) cudaFreeHost(e->h_newc);
    if (e->h_height) cudaFreeHost(e->h_height);
    if (e->h_seq) cudaFreeHost(e->h_seq);
    if (e->h_stale) cudaFreeHost(e->h_stale);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

int sw_reset(sw_engine *e) {
    if (!e) return SW_E_ARG;
    CK(cudaSetDevice(e->device));
    if (wait_appends(e, -1) < 0) return SW_E_CUDA;
    CK(cudaStreamSynchronize(e->stream));
    fold_spans(e);
    e->h_creator.clear();
    e->ids.clear();
    e->h_stale_cum.assign(1, 0);
    int rc = reset_state(e);
    memset(&e->stats, 0, sizeof e->stats);
    return rc;
}

int sw_rewind(sw_engine *e) {
    if (!e) return SW_E_ARG;
    CK(cudaSetDevice(e->device));
    if (wait_appends(e, -1) < 0) return SW_E_CUDA;
    CK(cudaStreamSynchronize(e->stream));
    fold_spans(e);
    return reset_state(e, true);
}

int sw_event_record(sw_engine *e, int slot) {
    if (!e || slot < 0 || slot >= 16) return fail(e, SW_E_ARG, "bad event slot");
    CK(cudaSetDevice(e->device));
    if (!e->user_ev[slot]) CK(cudaEventCreate(&e->user_ev[slot]));
    CK(cudaEventRecord(e->user_ev[slot], e->stream));
    return SW_OK;
}

int sw_event_elapsed_ms(sw_engine *e, int a, int b, double *ms_out) {
    if (!e || a < 0 || a >= 16 || b < 0 || b >= 16 || !ms_out || !e->user_ev[a] || !e->user_ev[b])
        return fail(e, SW_E_ARG, "bad event slot");
    CK(cudaSetDevice(e->device));
    CK(cudaEventSynchronize(e->user_ev[b]));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e->user_ev[a], e->user_ev[b]));
    *ms_out = ms;
    return SW_OK;
}

int sw_append(sw_engine *e, int n, const int32_t *p0, const int32_t *p1, const int32_t *creator,
              const double *t, const uint8_t *sig) {
    if (!e || n < 0 || (n > 0 && (!p0 || !p1 || !creator || !t || !sig))) return fail(e, SW_E_ARG, "bad argument");
    if (n == 0) return SW_OK;
    if ((i64)e->n_events + n > e->cap) return fail(e, SW_E_CAPACITY, "capacity_events=%d exceeded", e->cap);
    CK(cudaSetDevice(e->device));
    const int base = e->n_events;
    // graph-shape checks of is_valid_event (swirld.py:104-108) + the fork-free contract
    std::vector<int32_t> head_save(e->h_head), count_save(e->h_count);
    e->h_creator.resize((size_t)base + n);
    int rc = SW_OK;
    for (int j = 0; j < n && rc == SW_OK; j++) {
        const int i = base + j, c = creator[j], a = p0[j], b = p1[j];
        if (c < 0 || c >= e->M) { rc = fail(e, SW_E_ARG, "event %d: creator %d out of range", i, c); break; }
        e->h_stale[i] = 0;
        if (a < 0 && b < 0) {
            if (e->h_head[c] >= 0) { rc = fail(e, SW_E_FORK, "event %d: second root of member %d", i, c); break; }
            e->h_height[i] = 0;                                          // swirld.py:117-118
        } else {
            if (a < 0 || b < 0 || a >= i || b >= i) { rc = fail(e, SW_E_PARENT, "event %d: parents (%d,%d) unknown", i, a, b); break; }
            if (e->h_creator[a] != c) { rc = fail(e, SW_E_PARENT, "event %d: self-parent %d has another creator", i, a); break; }
            if (e->h_creator[b] == c) { rc = fail(e, SW_E_PARENT, "event %d: other-parent %d has the same creator", i, b); break; }
            if (e->h_head[c] != a) { rc = fail(e, SW_E_FORK, "event %d: self-parent %d is not member %d's latest event (fork)", i, a, c); break; }
            e->h_height[i] = std::max(e->h_height[a], e->h_height[b]) + 1;   // swirld.py:120
            e->h_stale[i] = e->h_head[e->h_creator[b]] != b;             // "near fork": an older event of the peer
        }
        e->h_creator[i] = c;
        e->h_head[c] = i;
        e->h_seq[i] = e->h_count[c]++;
    }
    if (rc == SW_OK) {
        e->h_stale_cum.resize((size_t)base + n + 1);
        for (int j = 0; j < n; j++) e->h_stale_cum[base + j + 1] = e->h_stale_cum[base + j] + e->h_stale[base + j];
    }
    if (rc != SW_OK) {
        e->h_head = head_save; e->h_count = count_save;
        e->h_creator.resize(base);
        return rc;
    }
    // The copies go to their own stream: they touch only the new rows, so they overlap the kernels of
    // earlier chunks still running on the compute stream; later compute work waits for them.
    cudaStream_t cs = e->copy_stream;
    if (n <= sw_engine::STAGE_EVENTS) {
        // a handful of events: pack the eight columns into one pinned block, one copy, one scatter kernel
        const size_t slot = (unpack_bytes(sw_engine::STAGE_EVENTS) + 255) & ~(size_t)255;
        const int si = e->stage_next;
        e->stage_next = (si + 1) % sw_engine::STAGE_SLOTS;
        CK(cudaEventSynchronize(e->stage_ev[si]));                       // (the copy that used this slot eight appends ago)
        uint8_t *hs = e->h_stage + slot * si, *ds = e->d_stage + slot * si;
        int32_t *ints = reinterpret_cast<int32_t *>(hs);
        memcpy(ints, p0, sizeof(int32_t) * n); memcpy(ints + n, p1, sizeof(int32_t) * n); memcpy(ints + 2 * n, creator, sizeof(int32_t) * n);
        memcpy(ints + 3 * n, e->h_seq + base, sizeof(int32_t) * n); memcpy(ints + 4 * n, e->h_height + base, sizeof(int32_t) * n);
        uint8_t *pt = hs + unpack_off_t(n);
        memcpy(pt, t, sizeof(double) * n); memcpy(pt + (size_t)8 * n, sig, (size_t)64 * n); memcpy(pt + (size_t)72 * n, e->h_stale + base, (size_t)n);
        CK(cudaMemcpyAsync(ds, hs, unpack_bytes(n), cudaMemcpyHostToDevice, cs));
        CK(cudaEventRecord(e->stage_ev[si], cs));
        UnpackParams U{};
        U.base = base; U.n = n; U.stage = ds; U.p0 = e->d_p0; U.p1 = e->d_p1; U.creator = e->d_creator; U.seq = e->d_seq;
        U.height = e->d_height; U.t = e->d_t; U.sig = e->d_sig; U.stale = e->d_stale;
        k_unpack<<<1, 256, 0, cs>>>(U);
        CK(cudaGetLastError());
        e->stats.kernel_launches += 1;
    } else {
        CK(cudaMemcpyAsync(e->d_p0 + base, p0, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_p1 + base, p1, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_creator + base, creator, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_t + base, t, sizeof(double) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_sig + (size_t)base * 64, sig, (size_t)64 * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_seq + base, e->h_seq + base, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_height + base, e->h_height + base, sizeof(int32_t) * n, cudaMemcpyHostToDevice, cs));
        CK(cudaMemcpyAsync(e->d_stale + base, e->h_stale + base, (size_t)n, cudaMemcpyHostToDevice, cs));
    }
    // rows are up to date and the batch is big: scan it now, beside the kernels of the previous chunk
    // (several ranks: the scan holds cross-GPU barriers; it must not run beside a round kernel that fills every SM while
    //  waiting for the same peer -- scans stay on the compute stream then)
    const bool eager = e->n_rowed == base && n >= 4096 && e->nranks == 1;
    e->stats.h2d_bytes += (i64)n * (5 * 4 + 1 + 8 + 64);
    e->stats.events += n;
    e->n_events += n;
    if (eager) {
        if (e->scan_ev_set) CK(cudaStreamWaitEvent(cs, e->scan_ev, 0));     // never beside a scan on the compute stream
        int rc2 = cansee_scan(e, cs, e->n_events);
        if (rc2 < 0) return rc2;
    }
    // the compute stream waits for this batch only when a call first touches it (wait_appends)
    cudaEvent_t done = get_event(e);
    CK(cudaEventRecord(done, cs));
    e->appends.push_back({base, done});
    return SW_OK;
}

int sw_divide_rounds(sw_engine *e, int first, int n) {
    if (!e || n < 0) return fail(e, SW_E_ARG, "bad argument");
    if (n == 0) return SW_OK;
    if (first != e->n_divided) return fail(e, SW_E_ARG, "divide_rounds: first=%d but %d events are divided (events must arrive in order)", first, e->n_divided);
    if (first + n > e->n_events) return fail(e, SW_E_KEY, "divide_rounds: events [%d,%d) not appended", first, first + n);
    CK(cudaSetDevice(e->device));
    if (n <= e->stream_n && e->n_rowed == first) {
        // the reference's own cadence (one sync per call): the whole of divide_rounds in ONE launch (swirld_stream.cuh)
        if (wait_appends(e, first + n) < 0) return SW_E_CUDA;
        const int M = e->M;
        StreamParams S{};
        S.M = M; S.first = first; S.n = n; S.Rcap = e->Rcap; S.NJ = e->NJ;
        S.p0 = e->d_p0; S.p1 = e->d_p1; S.creator = e->d_creator; S.seq = e->d_seq; S.row = e->d_row; S.round = e->d_round;
        S.wit = e->d_wit; S.W = e->d_W; S.Wf = e->d_Wf; S.SM = e->d_SM; S.S = e->d_S; S.SMw = e->d_SMw; S.Sw = e->d_Sw;
        S.coin = e->d_coin; S.sig = e->d_sig; S.stake = e->d_stake; S.tot2 = 2 * e->tot; S.scal = e->d_scal;
        S.ctot = e->d_rbtot; S.gchain = e->d_gchain; S.carry = e->d_cs_carry; S.ring = RB_RING;
        const int threads = std::min(1024, std::max(32, (M + 31) / 32 * 32));
        const size_t smem = (size_t)M * 8 + 32 * 8 + (size_t)3 * M * 4 + 32 * 4;
        {
            Span sp(e, 0);
            if (e->wide) k_stream_divide<true><<<1, threads, smem, e->stream>>>(S);
            else k_stream_divide<false><<<1, threads, smem, e->stream>>>(S);
            CK(cudaGetLastError());
        }
        e->n_rowed = first + n;
        CK(cudaEventRecord(e->scan_ev, e->stream));         // (it wrote can_see rows and the carry heads on the compute stream)
        e->scan_ev_set = true;
        e->stats.kernel_launches += 1;
        e->stats.events_divided += n;
        e->n_divided += n;
        return SW_OK;
    }
    if (first + n > e->n_rowed) {
        // rows are behind (small appends, or after sw_rewind): scan everything appended so far, here -- after the
        // copies of EVERY appended batch (the scan reads the columns of all of them)
        if (wait_appends(e, -1) < 0) return SW_E_CUDA;
        int rc = cansee_scan(e, e->stream, e->n_events);
        if (rc < 0) return rc;
        CK(cudaEventRecord(e->scan_ev, e->stream));
        e->scan_ev_set = true;
    } else if (wait_appends(e, first + n) < 0) return SW_E_CUDA;
    {
        Span sp(e, 0);
        int rc;
        if (e->wide) rc = SW_NJ(divide_rounds_wide, e, first, n);
        else rc = e->NC == 1 ? (e->unit ? divide_round_batch<1, true>(e, first, n) : divide_round_batch<1, false>(e, first, n))
                             : (e->unit ? divide_round_batch<2, true>(e, first, n) : divide_round_batch<2, false>(e, first, n));
        if (rc < 0) return rc;
    }
    e->stats.events_divided += n;
    e->n_divided += n;
    return SW_OK;
}

// Node.divide_rounds for B independent node-views at once (M <= 64, same member count, same device): everything of a
// view runs on the view's own stream, except the round kernels, which advance side by side in ONE cooperative launch.
int sw_batch_divide_rounds(sw_engine *const *engines, int B, const int *first, const int *n) {
    sw_engine *e = (engines && B > 0) ? engines[0] : nullptr;
    if (!e || !first || !n) return fail(e, SW_E_ARG, "bad argument");
    for (int v = 0; v < B; v++) {
        sw_engine *x = engines[v];
        if (!x || x->wide || x->M != e->M || x->device != e->device || x->unit != e->unit)
            return fail(e, SW_E_UNSUPPORTED, "sw_batch_divide_rounds: the views must be M <= 64 engines of one shape on one device");
        if (n[v] <= 0 || first[v] != x->n_divided || first[v] + n[v] > x->n_events)
            return fail(e, SW_E_ARG, "sw_batch_divide_rounds: view %d: bad range [%d,%d)", v, first[v], first[v] + n[v]);
    }
    CK(cudaSetDevice(e->device));
    const int gmin = 1;                                     // (a view's warps loop over its (chain, position) pairs)
    const int per_launch = std::max(1, e->n_sm / gmin);
    if (B > e->views_cap) {
        if (e->d_views) cudaFree(e->d_views);
        if (e->d_rcviews) cudaFree(e->d_rcviews);
        e->d_views = nullptr; e->d_rcviews = nullptr;
        CK(cudaMalloc((void **)&e->d_views, sizeof(RbParams) * B));
        CK(cudaMalloc((void **)&e->d_rcviews, sizeof(RcParams) * B));
        e->views_cap = B;
    }
    // one thread-block cluster per view first (swirld_rcluster.cuh); the grid-wide kernel then takes what they hand back
    bool use_rc = true;
    for (int v = 0; v < B; v++) use_rc = use_rc && engines[v]->rc_ok && engines[v]->rc_mb == e->rc_mb && n[v] >= e->rc_min_n;
    std::vector<RcParams> Qv(B);
    if (!e->view_ev) CK(cudaEventCreateWithFlags(&e->view_ev, cudaEventDisableTiming));
    std::vector<RbParams> Rv(B);
    for (int v0 = 0; v0 < B; v0 += per_launch) {
        const int nv = std::min(per_launch, B - v0), G = std::max(gmin, e->n_sm / nv);
        for (int v = v0; v < v0 + nv; v++) {
            sw_engine *x = engines[v];
            if (first[v] + n[v] > x->n_rowed) {
                if (wait_appends(x, -1) < 0) return SW_E_CUDA;
                if (cansee_scan(x, x->stream, x->n_events) < 0) return SW_E_CUDA;
                CK(cudaEventRecord(x->scan_ev, x->stream));
                x->scan_ev_set = true;
            } else if (wait_appends(x, first[v] + n[v]) < 0) return SW_E_CUDA;
            // a view's window stays a round deep (16 pending events per chain) however few warps it has: they loop
            if (round_batch_prep(x, first[v], n[v], G, Rv[v], 16) < 0) { e->err = x->err; return SW_E_CUDA; }
            if (use_rc) {
                if (rc_seqrows(x, Rv[v]) < 0) { e->err = x->err; return SW_E_CUDA; }
                Qv[v] = RcParams{Rv[v], x->d_rsg, x->d_rccont};
                Rv[v].cont = x->d_rccont;
                x->stats.kernel_launches += 1;
            }
            cudaEvent_t ev = get_event(x);
            CK(cudaEventRecord(ev, x->stream));
            CK(cudaStreamWaitEvent(e->stream, ev, 0));
            x->pool.push_back(ev);
        }
        CK(cudaMemcpyAsync(e->d_views + v0, Rv.data() + v0, sizeof(RbParams) * nv, cudaMemcpyHostToDevice, e->stream));
        const RbParams *pv = e->d_views + v0;
        int g = G;
        void *args[] = {(void *)&pv, (void *)&g};
        {
            cudaEvent_t a = get_event(e), b = get_event(e);
            cudaEventRecord(a, e->stream);
            if (use_rc) {
                CK(cudaMemcpyAsync(e->d_rcviews + v0, Qv.data() + v0, sizeof(RcParams) * nv, cudaMemcpyHostToDevice, e->stream));
                cudaLaunchConfig_t cfg;
                cudaLaunchAttribute at[1];
                rc_launch_config(cfg, at, nv, e->stream);
                const RcParams *qv = e->d_rcviews + v0;
                if (e->unit) { if (e->rc_mb) CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster_views<true, true>, qv)); else CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster_views<true, false>, qv)); }
                else { if (e->rc_mb) CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster_views<false, true>, qv)); else CK(cudaLaunchKernelEx(&cfg, k_rounds_cluster_views<false, false>, qv)); }
                e->stats.kernel_launches += 1;
            }
            void *fn = e->NC == 1 ? (e->unit ? (void *)k_rounds_batch_views<1, true> : (void *)k_rounds_batch_views<1, false>)
                                  : (e->unit ? (void *)k_rounds_batch_views<2, true> : (void *)k_rounds_batch_views<2, false>);
            CK(cudaLaunchCooperativeKernel(fn, dim3(nv * G), dim3(RB_THREADS), args, 0, e->stream));
            cudaEventRecord(b, e->stream);
            e->spans.push_back(TimedSpan{a, b, 4});
        }
        CK(cudaEventRecord(e->view_ev, e->stream));
        CK(cudaStreamSynchronize(e->stream));       // (Rv / the event are reused by the next group; the views' finish kernels follow)
        for (int v = v0; v < v0 + nv; v++) {
            sw_engine *x = engines[v];
            int rc = x->NC == 1 ? round_batch_finish<1>(x, Rv[v]) : round_batch_finish<2>(x, Rv[v]);
            if (rc < 0) return rc;
            x->stats.events_divided += n[v];
            x->n_divided += n[v];
        }
    }
    return SW_OK;
}

int sw_decide_fame(sw_engine *e, int32_t *new_c_out, int cap) {
    if (!e || cap < 0 || (cap > 0 && !new_c_out)) return fail(e, SW_E_ARG, "bad argument");
    CK(cudaSetDevice(e->device));
    if (e->n_divided == 0) return fail(e, SW_E_ARG, "decide_fame: no witnesses yet (max() of an empty dict, swirld.py:225)");
    FameParams P{};
    P.M = e->M; P.Rcap = e->Rcap; P.C = e->C; P.W = e->d_W; P.S = e->d_S; P.famous = e->d_famous;
    P.famous_ev = e->d_famous_ev; P.consensus = e->d_consensus; P.done = e->d_done; P.rem = e->d_rem;
    P.coin = e->d_coin; P.stake = e->d_stake; P.tot2 = 2 * e->tot; P.unit = e->unit ? 1 : 0; P.newc = e->d_newc; P.scal = e->d_scal;
    P.Sw = e->d_Sw;
    {
        Span sp(e, 1);
        k_fame_begin<<<1, 32, 0, e->stream>>>(P);
        if (e->wide) SW_NJ(fame_rounds_wide, e, P);
        else k_fame_rounds<<<2 * e->n_sm, 256, 0, e->stream>>>(P);
        k_fame_finish<<<1, 1024, 0, e->stream>>>(P);
        CK(cudaGetLastError());
    }
    e->stats.kernel_launches += 3;
    // one copy pair, one synchronisation: the scalars and (speculatively) the first new consensus rounds together
    const int spec = std::min(e->Rcap, 64);
    CK(cudaMemcpyAsync(e->h_scal, e->d_scal, sizeof(int32_t) * SC_COUNT, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaMemcpyAsync(e->h_newc, e->d_newc, sizeof(int32_t) * spec, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    fold_spans(e);
    e->stats.d2h_bytes += sizeof(int32_t) * (SC_COUNT + spec);
    int rc = device_error(e);
    if (rc < 0) return rc;
    const int cnt = e->h_scal[SC_NEWC];
    if (cnt > cap) return fail(e, SW_E_ARG, "decide_fame: %d new consensus rounds do not fit cap=%d", cnt, cap);
    if (cnt > spec) {
        CK(cudaMemcpyAsync(e->h_newc, e->d_newc, sizeof(int32_t) * cnt, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        e->stats.d2h_bytes += sizeof(int32_t) * cnt;
    }
    if (cnt > 0) memcpy(new_c_out, e->h_newc, sizeof(int32_t) * cnt);
    return cnt;
}

int sw_find_order(sw_engine *e, const int32_t *new_c, int n) {
    if (!e || n < 0 || (n > 0 && !new_c)) return fail(e, SW_E_ARG, "bad argument");
    if (n == 0) return 0;
    CK(cudaSetDevice(e->device));
    std::vector<int32_t> rs(new_c, new_c + n);
    std::sort(rs.begin(), rs.end());                                  // sorted(new_c), swirld.py:283
    for (int r : rs) if (r < 0 || r >= e->Rcap) return fail(e, SW_E_KEY, "find_order: unknown round %d", r);
    const size_t MS = e->MS;
    if (n > e->seg_cap) {
        int nc = std::max(n, std::max(64, 2 * e->seg_cap));
        for (void *p : {(void *)e->d_seg_start, (void *)e->d_seg_fw, (void *)e->d_seg_nf, (void *)e->d_seg_white, (void *)e->d_rounds_in, (void *)e->d_plan})
            if (p) cudaFree(p);
        CK(dalloc(&e->d_seg_start, (size_t)nc + 1)); CK(dalloc(&e->d_seg_fw, (size_t)nc * MS));
        CK(dalloc(&e->d_seg_nf, (size_t)nc)); CK(dalloc(&e->d_seg_white, (size_t)nc * 64));
        CK(dalloc(&e->d_rounds_in, (size_t)nc)); CK(dalloc(&e->d_plan, (size_t)nc * MS * 8));
        e->seg_cap = nc;
    }
    CK(cudaMemcpyAsync(e->d_rounds_in, rs.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, e->stream));
    OrderParams P{};
    P.M = e->M; P.Rcap = e->Rcap; P.nrounds = n; P.rounds = e->d_rounds_in; P.W = e->d_W; P.famous = e->d_famous;
    P.row = e->d_row; P.p0 = e->d_p0; P.creator = e->d_creator; P.seq = e->d_seq; P.t = e->d_t; P.sig = e->d_sig;
    P.stake = e->d_stake; P.tot = e->tot; P.lastord = e->d_lastord; P.batch_ev = e->d_batch_ev; P.batch_seg = e->d_batch_seg;
    P.seg_start = e->d_seg_start; P.seg_fw = e->d_seg_fw; P.seg_nf = e->d_seg_nf; P.seg_white = e->d_seg_white;
    P.ts = e->d_ts; P.key = e->d_key; P.perm = e->d_perm; P.tx = e->d_tx; P.idx = e->d_idx; P.tx_base = e->n_tx; P.scal = e->d_scal;
    P.plan = e->d_plan; P.plan_stride = (int)(e->seg_cap * MS);
    const int M = e->M;
    cudaEvent_t a = get_event(e), b = get_event(e);
    cudaEventRecord(a, e->stream);
    if (e->wide) {
        k_w_order_rounds<<<n, 1024, (size_t)3 * M * sizeof(int), e->stream>>>(P);
        k_w_order_cuts<<<1, 1024, (size_t)2 * M * sizeof(int), e->stream>>>(P);
        k_w_order_list<<<std::max(1, std::min(4 * e->n_sm, (int)(((size_t)n * M + 255) / 256))), 256, 0, e->stream>>>(P);
    } else {
        k_order_rounds<<<n, 1024, 0, e->stream>>>(P);
        k_order_cuts<<<1, 64, 0, e->stream>>>(P);
        k_order_list<<<std::max(1, std::min(4 * e->n_sm, (n * 64 + 255) / 256)), 256, 0, e->stream>>>(P);
    }
    CK(cudaGetLastError());
    // the number of newly ordered events stays on the device: the time / sort kernels read it there, the host learns it
    // from the one copy at the end of the call
    if (e->wide) {
        const size_t tsm = (size_t)OW_WARPS * M * sizeof(u64);
        k_w_order_times<<<8 * e->n_sm, OW_WARPS * 32, tsm, e->stream>>>(P);
    } else k_order_times<<<4 * e->n_sm, 256, 0, e->stream>>>(P);
    k_order_sort<<<n, 1024, 0, e->stream>>>(P);
    CK(cudaGetLastError());
    cudaEventRecord(b, e->stream);
    e->spans.push_back(TimedSpan{a, b, 2});
    CK(cudaMemcpyAsync(e->h_scal, e->d_scal, sizeof(int32_t) * SC_COUNT, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));      // (rs, the host vector of the rounds, was consumed by the copy above)
    fold_spans(e);
    e->stats.kernel_launches += 5;
    e->stats.h2d_bytes += sizeof(int32_t) * n;
    e->stats.d2h_bytes += sizeof(int32_t) * SC_COUNT;
    int rc = device_error(e);
    if (rc < 0) return rc;
    const int nbatch = e->h_scal[SC_BATCH];
    e->n_tx += nbatch;
    return nbatch;
}

int sw_members(const sw_engine *e) { return e ? e->M : SW_E_ARG; }
int sw_n_events(const sw_engine *e) { return e ? e->n_events : SW_E_ARG; }
int sw_n_divided(const sw_engine *e) { return e ? e->n_divided : SW_E_ARG; }
int sw_n_transactions(const sw_engine *e) { return e ? e->n_tx : SW_E_ARG; }

int sw_sync(sw_engine *e) {
    if (!e) return SW_E_ARG;
    CK(cudaSetDevice(e->device));
    if (wait_appends(e, -1) < 0) return SW_E_CUDA;
    CK(cudaMemcpyAsync(e->h_scal, e->d_scal, sizeof(int32_t) * SC_COUNT, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    fold_spans(e);
    return device_error(e);
}

int sw_max_round(sw_engine *e) {
    int rc = sw_sync(e);
    if (rc < 0) return rc;
    return e->h_scal[SC_MAX_ROUND];
}

int sw_stats(sw_engine *e, sw_stats_t *out) {
    if (!e || !out) return SW_E_ARG;
    int rc = sw_sync(e);
    *out = e->stats;
    return rc;
}

#define GETTER(NAME, TYPE, SRC, LIMIT, WIDTH)                                                        \
    int NAME(sw_engine *e, int first, int n, TYPE *out) {                                            \
        if (!e || first < 0 || n < 0 || (n > 0 && !out)) return fail(e, SW_E_ARG, "bad argument");  \
        if (first + n > (LIMIT)) return fail(e, SW_E_KEY, #NAME ": [%d,%d) out of range", first, first + n); \
        if (n == 0) return SW_OK;                                                                    \
        CK(cudaSetDevice(e->device));                                                                \
        if (wait_appends(e, -1) < 0) return SW_E_CUDA;                                               \
        CK(cudaMemcpyAsync(out, (SRC) + (size_t)first * (WIDTH), sizeof(TYPE) * (size_t)n * (WIDTH), \
                           cudaMemcpyDeviceToHost, e->stream));                                     \
        CK(cudaStreamSynchronize(e->stream));                                                        \
        e->stats.d2h_bytes += sizeof(TYPE) * (size_t)n * (WIDTH);                                    \
        return SW_OK;                                                                                \
    }

GETTER(sw_get_round, int32_t, e->d_round, e->n_divided, 1)
GETTER(sw_get_witness_flags, uint8_t, e->d_wit, e->n_divided, 1)
GETTER(sw_get_famous, int8_t, e->d_famous_ev, e->n_events, 1)
GETTER(sw_get_can_see, int32_t, e->d_row, e->n_divided, e->M)
GETTER(sw_get_witness_table, int32_t, e->d_W, e->Rcap, e->M)
GETTER(sw_get_transactions, int32_t, e->d_tx, e->n_tx, 1)
GETTER(sw_get_idx, int32_t, e->d_idx, e->n_events, 1)

int sw_get_height(sw_engine *e, int first, int n, int32_t *out) {
    if (!e || first < 0 || n < 0 || (n > 0 && !out)) return fail(e, SW_E_ARG, "bad argument");
    if (first + n > e->n_events) return fail(e, SW_E_KEY, "sw_get_height: out of range");
    memcpy(out, e->h_height + first, sizeof(int32_t) * n);
    return SW_OK;
}

int sw_get_consensus(sw_engine *e, int32_t *out, int cap) {
    if (!e || cap < 0) return fail(e, SW_E_ARG, "bad argument");
    int mr = sw_max_round(e);
    if (mr < -1) return mr;
    std::vector<uint8_t> flags((size_t)mr + 2);
    if (mr >= 0) {
        CK(cudaMemcpyAsync(flags.data(), e->d_consensus, (size_t)mr + 1, cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        e->stats.d2h_bytes += mr + 1;
    }
    int cnt = 0;
    for (int r = 0; r <= mr; r++)
        if (flags[r]) { if (cnt < cap) out[cnt] = r; cnt++; }
    return cnt;
}

int sw_debug_counters(sw_engine *e, int64_t *out16, int clear) {
    if (!e || !out16) return SW_E_ARG;
    CK(cudaSetDevice(e->device));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(out16, e->d_dbg, sizeof(long long) * 16, cudaMemcpyDeviceToHost));
    if (clear) CK(cudaMemset(e->d_dbg, 0, sizeof(long long) * 40));
    return SW_OK;
}

int sw_flush_l2(sw_engine *e, int64_t bytes) {
    if (!e || bytes <= 0) return SW_E_ARG;
    CK(cudaSetDevice(e->device));
    if ((size_t)bytes > e->flush_bytes) {
        if (e->d_flush) cudaFree(e->d_flush);
        e->d_flush = nullptr;
        CK(cudaMalloc(&e->d_flush, (size_t)bytes));
        e->flush_bytes = (size_t)bytes;
    }
    CK(cudaMemsetAsync(e->d_flush, 0x5a, (size_t)bytes, e->stream));
    return SW_OK;
}

// ---- ingest: what Node.sync does between the wire and divide_rounds (swirld.py:129-136, utils.py:8-21), natively.
// rejected (optional): input events that failed a check made before (the crypto checks of sw_ingest_verified); they
// are skipped like a shape- or fork-invalid event, and so is whatever hangs below them.
namespace {
int ingest_impl(sw_engine *e, int n, const uint8_t *ids, const uint8_t *p0_ids, const uint8_t *p1_ids,
                const int32_t *creator, const double *t, const uint8_t *sig, const uint8_t *rejected, int32_t *index_out) {
    auto key = [](const uint8_t *p) { Id32 k; memcpy(k.data(), p, 32); return k; };
    const Id32 zero{};
    // 1. which events are new, and where each new id sits in the batch
    std::unordered_map<Id32, int, Id32Hash> inbatch;
    inbatch.reserve((size_t)n * 2);
    for (int i = 0; i < n; i++) {
        const Id32 k = key(ids + (size_t)32 * i);
        auto it = e->ids.find(k);
        if (it != e->ids.end()) index_out[i] = it->second;
        else { index_out[i] = -1; inbatch.emplace(k, i); }       // (a duplicate id in the batch: the first one counts)
    }
    // 2. parents-first order of the new ones (iterative DFS; the edges are the parents that are in the batch)
    std::vector<int> order, state(n, 0);                           // 0 unseen, 1 on the stack, 2 done
    order.reserve(inbatch.size());
    std::vector<std::pair<int, int>> stack;
    auto parent_in_batch = [&](int i, int which) -> int {
        const Id32 k = key((which ? p1_ids : p0_ids) + (size_t)32 * i);
        if (k == zero) return -1;
        auto it = inbatch.find(k);
        return it == inbatch.end() ? -1 : it->second;
    };
    for (int r = 0; r < n; r++) {
        if (index_out[r] >= 0 || state[r] || inbatch.find(key(ids + (size_t)32 * r))->second != r) continue;
        stack.push_back({r, 0});
        state[r] = 1;
        while (!stack.empty()) {
            auto &[u, next] = stack.back();
            if (next < 2) {
                const int v = parent_in_batch(u, next++);
                if (v < 0 || state[v] == 2) continue;
                if (state[v] == 1) return fail(e, SW_E_ARG, "sw_ingest: the batch is not a DAG (utils.py:13)");
                state[v] = 1;
                stack.push_back({v, 0});
            } else { state[u] = 2; order.push_back(u); stack.pop_back(); }
        }
    }
    // 3. validate in that order against a scratch copy of the chain heads; what fails (and what hangs below it) is skipped
    std::vector<int32_t> head(e->h_head), bidx(n, -1), bcreator;
    std::vector<int32_t> c_p0, c_p1, c_cr, src;
    std::vector<double> c_t;
    int next_index = e->n_events;
    auto resolve = [&](int i, int which, int &out) -> bool {        // parent id -> arrival index (-1: no parent)
        const Id32 k = key((which ? p1_ids : p0_ids) + (size_t)32 * i);
        if (k == zero) { out = -1; return true; }
        auto g = e->ids.find(k);
        if (g != e->ids.end()) { out = g->second; return true; }
        auto b = inbatch.find(k);
        if (b != inbatch.end() && bidx[b->second] >= 0) { out = bidx[b->second]; return true; }
        return false;
    };
    auto creator_of = [&](int idx) { return idx < e->n_events ? e->h_creator[idx] : bcreator[idx - e->n_events]; };
    for (int i : order) {
        const int c = creator[i];
        int a, b;
        if ((rejected && rejected[i]) || c < 0 || c >= e->M || !resolve(i, 0, a) || !resolve(i, 1, b)) continue;
        if (a < 0 && b < 0) { if (head[c] >= 0) continue; }                         // a second root: fork
        else if (a < 0 || b < 0 || creator_of(a) != c || creator_of(b) == c || head[c] != a) continue;   // swirld.py:104-108 + fork-free
        if (next_index >= e->cap) return fail(e, SW_E_CAPACITY, "capacity_events=%d exceeded", e->cap);
        bidx[i] = next_index++;
        head[c] = bidx[i];
        bcreator.push_back(c);
        c_p0.push_back(a); c_p1.push_back(b); c_cr.push_back(c); c_t.push_back(t[i]); src.push_back(i);
    }
    // 4. one sw_append for the accepted events, then the ids
    const int m = (int)src.size();
    if (m > 0) {
        std::vector<uint8_t> c_sig((size_t)64 * m);
        for (int j = 0; j < m; j++) memcpy(c_sig.data() + (size_t)64 * j, sig + (size_t)64 * src[j], 64);
        int rc = sw_append(e, m, c_p0.data(), c_p1.data(), c_cr.data(), c_t.data(), c_sig.data());
        if (rc < 0) return rc;
        // (pageable sources: the copies are staged before sw_append returns, the vectors may go)
        CK(cudaStreamSynchronize(e->copy_stream));
        for (int j = 0; j < m; j++) e->ids.emplace(key(ids + (size_t)32 * src[j]), bidx[src[j]]);
    }
    for (int i = 0; i < n; i++)
        if (index_out[i] < 0) { auto it = e->ids.find(key(ids + (size_t)32 * i)); index_out[i] = it == e->ids.end() ? -1 : it->second; }
    return m;
}
}  // namespace

int sw_ingest(sw_engine *e, int n, const uint8_t *ids, const uint8_t *p0_ids, const uint8_t *p1_ids,
              const int32_t *creator, const double *t, const uint8_t *sig, int32_t *index_out) {
    if (!e || n < 0 || (n > 0 && (!ids || !p0_ids || !p1_ids || !creator || !t || !sig || !index_out))) return fail(e, SW_E_ARG, "bad argument");
    return ingest_impl(e, n, ids, p0_ids, p1_ids, creator, t, sig, nullptr, index_out);
}

// ---- is_valid_event's crypto checks (swirld.py:97-103) on the device: swirld_verify.cuh
int sw_set_member_keys(sw_engine *e, const uint8_t *pk) {
    if (!e || !pk) return fail(e, SW_E_ARG, "bad argument");
    CK(cudaSetDevice(e->device));
    const int M = e->M;
    if (!e->d_vtab) {
        CK(dalloc(&e->d_vpk, (size_t)32 * M));
        CK(dalloc(&e->d_vkeyok, (size_t)M + 1));
        CK(dalloc(&e->d_vbase, (size_t)M + 1));
        CK(dalloc(&e->d_vtab, (size_t)(M + 1) * swv::COMB_ENTRIES));
    }
    e->keys_set = false;
    CK(cudaMemcpyAsync(e->d_vpk, pk, (size_t)32 * M, cudaMemcpyHostToDevice, e->stream));
    k_verify_keys<<<(M + 1 + 127) / 128, 128, 0, e->stream>>>(e->d_vpk, M, e->d_vbase, e->d_vkeyok);
    k_verify_table<<<((M + 1) * 64 + 127) / 128, 128, 0, e->stream>>>(e->d_vbase, e->d_vkeyok, M, e->d_vtab);
    CK(cudaGetLastError());
    std::vector<uint8_t> ok((size_t)M + 1);
    CK(cudaMemcpyAsync(ok.data(), e->d_vkeyok, (size_t)M + 1, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->stats.kernel_launches += 2;
    e->stats.h2d_bytes += (int64_t)32 * M;
    e->stats.d2h_bytes += M + 1;
    if (!ok[M]) return fail(e, SW_E_CUDA, "sw_set_member_keys: the base point did not decode");
    e->keys_set = true;
    int bad = 0;
    for (int m = 0; m < M; m++) bad += ok[m] == 0;
    return bad;
}

namespace {
// the engine's grow-only scratch slot `slot`, at least `bytes` long
void *scratch(sw_engine *e, int slot, size_t bytes) {
    auto &b = e->vbuf[slot];
    bytes = std::max<size_t>(bytes, 16);
    if (bytes > b.cap) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr; b.cap = 0;
        if (cudaMalloc(&b.p, bytes + bytes / 4) != cudaSuccess) { b.p = nullptr; return nullptr; }
        b.cap = bytes + bytes / 4;
    }
    return b.p;
}

// device copy of a host buffer, in scratch slot `slot`
extern "C++" template <typename T>
int upload(sw_engine *e, int slot, const T *src, size_t count, const T **dst) {
    void *p = scratch(e, slot, count * sizeof(T));
    if (!p) return fail(e, SW_E_CUDA, "sw_verify: out of device memory for %zu bytes", count * sizeof(T));
    if (count) {
        CK(cudaMemcpyAsync(p, src, count * sizeof(T), cudaMemcpyHostToDevice, e->stream));
        e->stats.h2d_bytes += count * sizeof(T);
    }
    *dst = reinterpret_cast<const T *>(p);
    return 0;
}

bool offsets_ok(int n, const int64_t *off) {
    if (off[0] < 0) return false;
    for (int i = 0; i < n; i++) if (off[i + 1] < off[i]) return false;
    return true;
}

// status_out[i] for the events sel[0..nsel) (every event: sel NULL, nsel = n); the others' status is 0
int verify_impl(sw_engine *e, int n, const int32_t *sel, int nsel, const int32_t *creator, const uint8_t *sig,
                const uint8_t *msg, const int64_t *msg_off, const uint8_t *ids, const uint8_t *wire,
                const int64_t *wire_off, uint8_t *status_out) {
    if (!e->keys_set) return fail(e, SW_E_ARG, "sw_verify: call sw_set_member_keys first");
    if (!offsets_ok(n, msg_off) || !offsets_ok(n, wire_off)) return fail(e, SW_E_ARG, "sw_verify: offsets must start at >= 0 and not decrease");
    CK(cudaSetDevice(e->device));
    if (e->v_grid == 0) {
        CK(cudaFuncSetAttribute(k_verify, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(swv::Precomp) * swv::COMB_ENTRIES)));
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_verify, SWV_THREADS, sizeof(swv::Precomp) * swv::COMB_ENTRIES));
        e->v_grid = std::max(1, per_sm) * e->n_sm;
    }
    SwVerifyArgs a{};
    a.n = nsel; a.M = e->M;
    a.pk = e->d_vpk; a.keyok = e->d_vkeyok; a.tab = e->d_vtab;
    if (upload(e, 0, creator, (size_t)n, &a.creator) < 0 || upload(e, 1, sig, (size_t)64 * n, &a.sig) < 0 ||
        upload(e, 2, msg, (size_t)msg_off[n], &a.msg) < 0 || upload(e, 3, msg_off, (size_t)n + 1, &a.msg_off) < 0 ||
        upload(e, 4, ids, (size_t)32 * n, &a.ids) < 0 || upload(e, 5, wire, (size_t)wire_off[n], &a.wire) < 0 ||
        upload(e, 6, wire_off, (size_t)n + 1, &a.wire_off) < 0 || (sel && upload(e, 7, sel, (size_t)nsel, &a.sel) < 0))
        return SW_E_CUDA;
    uint8_t *d_status = reinterpret_cast<uint8_t *>(scratch(e, 8, (size_t)n));
    if (!d_status) return fail(e, SW_E_CUDA, "sw_verify: out of device memory");
    a.status = d_status;
    CK(cudaMemsetAsync(d_status, 0, (size_t)n, e->stream));
    if (nsel > 0) {
        const int grid = std::min(e->v_grid, (nsel + SWV_THREADS - 1) / SWV_THREADS);
        k_verify<<<grid, SWV_THREADS, sizeof(swv::Precomp) * swv::COMB_ENTRIES, e->stream>>>(a);
        CK(cudaGetLastError());
        e->stats.kernel_launches += 1;
    }
    CK(cudaMemcpyAsync(status_out, d_status, (size_t)n, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    e->stats.d2h_bytes += n;
    int good = 0;
    for (int i = 0; i < n; i++) good += status_out[i] == 3;
    return good;
}
}  // namespace

int sw_verify(sw_engine *e, int n, const int32_t *creator, const uint8_t *sig, const uint8_t *msg, const int64_t *msg_off,
              const uint8_t *ids, const uint8_t *wire, const int64_t *wire_off, uint8_t *status_out) {
    if (!e || n < 0 || !msg_off || !wire_off || (n > 0 && (!creator || !sig || !ids || !status_out)) ||
        (msg_off[n] > msg_off[0] && !msg) || (wire_off[n] > wire_off[0] && !wire))
        return fail(e, SW_E_ARG, "bad argument");
    return verify_impl(e, n, nullptr, n, creator, sig, msg, msg_off, ids, wire, wire_off, status_out);
}

int sw_ingest_verified(sw_engine *e, int n, const uint8_t *ids, const uint8_t *p0_ids, const uint8_t *p1_ids,
                       const int32_t *creator, const double *t, const uint8_t *sig, const uint8_t *msg,
                       const int64_t *msg_off, const uint8_t *wire, const int64_t *wire_off, int32_t *index_out) {
    if (!e || n < 0 || !msg_off || !wire_off ||
        (n > 0 && (!ids || !p0_ids || !p1_ids || !creator || !t || !sig || !index_out)) ||
        (msg_off[n] > msg_off[0] && !msg) || (wire_off[n] > wire_off[0] && !wire))
        return fail(e, SW_E_ARG, "bad argument");
    if (!e->keys_set) return fail(e, SW_E_ARG, "sw_ingest_verified: call sw_set_member_keys first");
    // only the events new to the engine are checked (ingest skips the known ones)
    std::vector<int32_t> sel;
    for (int i = 0; i < n; i++) {
        Id32 k;
        memcpy(k.data(), ids + (size_t)32 * i, 32);
        if (e->ids.find(k) == e->ids.end()) sel.push_back(i);
    }
    std::vector<uint8_t> status((size_t)n, 0), rejected((size_t)n, 0);
    if (!sel.empty()) {
        const int rc = verify_impl(e, n, sel.data(), (int)sel.size(), creator, sig, msg, msg_off, ids, wire, wire_off, status.data());
        if (rc < 0) return rc;
    }
    for (int i : sel) rejected[i] = status[i] != 3;
    return ingest_impl(e, n, ids, p0_ids, p1_ids, creator, t, sig, rejected.data(), index_out);
}

int sw_lookup(sw_engine *e, int n, const uint8_t *ids, int32_t *index_out) {
    if (!e || n < 0 || (n > 0 && (!ids || !index_out))) return fail(e, SW_E_ARG, "bad argument");
    for (int i = 0; i < n; i++) {
        Id32 k;
        memcpy(k.data(), ids + (size_t)32 * i, 32);
        auto it = e->ids.find(k);
        index_out[i] = it == e->ids.end() ? -1 : it->second;
    }
    return SW_OK;
}

// ---- checkpoint / resume: the engine's whole state as one binary file (sections of SoA columns)
namespace {
struct CkptHeader {
    char magic[8];
    int32_t version, M, cap, C, Rcap, wide, NJ, n_events, n_divided, n_tx, n_rowed, rounds;
    uint32_t rb_epoch, n_ids;
};
const char CKPT_MAGIC[8] = {'S', 'W', 'B', '2', 'C', 'K', 'P', 'T'};

bool put_host(FILE *f, const void *p, size_t bytes) {
    uint64_t nb = bytes;
    return fwrite(&nb, 8, 1, f) == 1 && (bytes == 0 || fwrite(p, 1, bytes, f) == bytes);
}
bool put_dev(sw_engine *e, FILE *f, const void *d, size_t bytes, std::vector<char> &tmp) {
    uint64_t nb = bytes;
    if (fwrite(&nb, 8, 1, f) != 1) return false;
    const size_t CH = (size_t)64 << 20;
    for (size_t o = 0; o < bytes; o += CH) {
        const size_t k = std::min(CH, bytes - o);
        tmp.resize(k);
        if (cudaMemcpyAsync(tmp.data(), (const char *)d + o, k, cudaMemcpyDeviceToHost, e->stream) != cudaSuccess) return false;
        if (cudaStreamSynchronize(e->stream) != cudaSuccess) return false;
        if (fwrite(tmp.data(), 1, k, f) != k) return false;
    }
    return true;
}
bool get_host(FILE *f, void *p, size_t bytes) {
    uint64_t nb = 0;
    return fread(&nb, 8, 1, f) == 1 && nb == bytes && (bytes == 0 || fread(p, 1, bytes, f) == bytes);
}
bool get_dev(sw_engine *e, FILE *f, void *d, size_t bytes, std::vector<char> &tmp) {
    uint64_t nb = 0;
    if (fread(&nb, 8, 1, f) != 1 || nb != bytes) return false;
    const size_t CH = (size_t)64 << 20;
    for (size_t o = 0; o < bytes; o += CH) {
        const size_t k = std::min(CH, bytes - o);
        tmp.resize(k);
        if (fread(tmp.data(), 1, k, f) != k) return false;
        if (cudaMemcpyAsync((char *)d + o, tmp.data(), k, cudaMemcpyHostToDevice, e->stream) != cudaSuccess) return false;
        if (cudaStreamSynchronize(e->stream) != cudaSuccess) return false;
    }
    return true;
}
}  // namespace

int sw_save(sw_engine *e, const char *path) {
    if (!e || !path) return fail(e, SW_E_ARG, "bad argument");
    if (e->nranks > 1) return fail(e, SW_E_UNSUPPORTED, "sw_save: checkpoint one rank of a multi-GPU engine is not supported");
    int rc = sw_sync(e);
    if (rc < 0) return rc;
    FILE *f = fopen(path, "wb");
    if (!f) return fail(e, SW_E_ARG, "sw_save: cannot open %s", path);
    const int M = e->M, n = e->n_events, nd = e->n_divided, nr = e->n_rowed;
    const int R = std::min(e->Rcap, e->h_scal[SC_MAX_ROUND] + 2);
    CkptHeader H{};
    memcpy(H.magic, CKPT_MAGIC, 8);
    H.version = 1; H.M = M; H.cap = e->cap; H.C = e->C; H.Rcap = e->Rcap; H.wide = e->wide ? 1 : 0; H.NJ = e->NJ;
    H.n_events = n; H.n_divided = nd; H.n_tx = e->n_tx; H.n_rowed = nr; H.rounds = R; H.rb_epoch = e->rb_epoch;
    H.n_ids = (uint32_t)e->ids.size();
    std::vector<uint8_t> idrec((size_t)36 * e->ids.size());
    { size_t o = 0; for (auto &kv : e->ids) { memcpy(&idrec[o], kv.first.data(), 32); memcpy(&idrec[o + 32], &kv.second, 4); o += 36; } }
    std::vector<char> tmp;
    const size_t RM = (size_t)R * M;
    bool ok = fwrite(&H, sizeof H, 1, f) == 1 && put_host(f, e->h_stake.data(), sizeof(i64) * M)
        && put_host(f, e->h_creator.data(), sizeof(int32_t) * n) && put_host(f, e->h_head.data(), sizeof(int32_t) * M)
        && put_host(f, e->h_count.data(), sizeof(int32_t) * M) && put_host(f, e->h_height, sizeof(int32_t) * n)
        && put_host(f, e->h_seq, sizeof(int32_t) * n) && put_host(f, e->h_stale, (size_t)n)
        && put_dev(e, f, e->d_p0, sizeof(int32_t) * n, tmp) && put_dev(e, f, e->d_p1, sizeof(int32_t) * n, tmp)
        && put_dev(e, f, e->d_creator, sizeof(int32_t) * n, tmp) && put_dev(e, f, e->d_t, sizeof(double) * n, tmp)
        && put_dev(e, f, e->d_sig, (size_t)64 * n, tmp)
        && put_dev(e, f, e->d_row, sizeof(int32_t) * (size_t)nr * M, tmp)
        && put_dev(e, f, e->d_round, sizeof(int32_t) * nd, tmp) && put_dev(e, f, e->d_wit, (size_t)nd, tmp)
        && (e->wide ? put_dev(e, f, e->d_SMw, sizeof(unsigned) * (size_t)nd * e->NJ, tmp) : put_dev(e, f, e->d_SM, sizeof(u64) * nd, tmp))
        && put_dev(e, f, e->d_famous_ev, (size_t)n, tmp) && put_dev(e, f, e->d_idx, sizeof(int32_t) * n, tmp)
        && put_dev(e, f, e->d_tx, sizeof(int32_t) * e->n_tx, tmp)
        && put_dev(e, f, e->d_W, sizeof(int32_t) * RM, tmp) && put_dev(e, f, e->d_Wf, sizeof(int32_t) * RM, tmp)
        && put_dev(e, f, e->d_famous, RM, tmp) && put_dev(e, f, e->d_coin, RM, tmp)
        && (e->wide ? put_dev(e, f, e->d_Sw, sizeof(unsigned) * RM * e->NJ, tmp) : put_dev(e, f, e->d_S, sizeof(u64) * RM, tmp))
        && put_dev(e, f, e->d_consensus, (size_t)R, tmp)
        && put_dev(e, f, e->d_lastord, sizeof(int32_t) * M, tmp) && put_dev(e, f, e->d_cs_carry, sizeof(int32_t) * M, tmp)
        && put_dev(e, f, e->d_rbtot, sizeof(int32_t) * M, tmp) && put_dev(e, f, e->d_gchain, sizeof(int32_t) * (size_t)M * RB_RING, tmp)
        && put_dev(e, f, e->d_scal, sizeof(int32_t) * SC_COUNT, tmp) && put_host(f, idrec.data(), idrec.size());
    ok = (fclose(f) == 0) && ok;
    if (!ok) return fail(e, SW_E_ARG, "sw_save: write to %s failed", path);
    return SW_OK;
}

int sw_load(const char *path, int device, int capacity_events, sw_engine **out) {
    sw_engine *e = nullptr;
    if (!path || !out) return fail(e, SW_E_ARG, "bad argument");
    *out = nullptr;
    FILE *f = fopen(path, "rb");
    if (!f) return fail(e, SW_E_ARG, "sw_load: cannot open %s", path);
    CkptHeader H{};
    if (fread(&H, sizeof H, 1, f) != 1 || memcmp(H.magic, CKPT_MAGIC, 8) != 0 || H.version != 1 || H.M < 1 || H.M > SW_MAX_MEMBERS) {
        fclose(f);
        return fail(e, SW_E_ARG, "sw_load: %s is not a swirld_b200 checkpoint", path);
    }
    std::vector<i64> stake(H.M);
    if (!get_host(f, stake.data(), sizeof(i64) * H.M)) { fclose(f); return fail(e, SW_E_ARG, "sw_load: truncated file"); }
    const int cap = std::max(capacity_events > 0 ? capacity_events : H.cap, H.n_events);
    // the saved engine's path (wide or not) is restored whatever SW_FORCE_WIDE says now
    setenv("SW_FORCE_WIDE", H.wide ? "1" : "0", 1);
    int rc = sw_create(H.M, cap, reinterpret_cast<const int64_t *>(stake.data()), H.C, device, &e);
    unsetenv("SW_FORCE_WIDE");
    if (rc < 0) { fclose(f); return rc; }
    const int M = H.M, n = H.n_events, nd = H.n_divided, nr = H.n_rowed, R = H.rounds;
    if (R > e->Rcap || (int)e->wide != H.wide || e->NJ != H.NJ) { fclose(f); sw_destroy(e); return fail(nullptr, SW_E_ARG, "sw_load: checkpoint does not fit the engine"); }
    std::vector<char> tmp;
    const size_t RM = (size_t)R * M;
    e->h_creator.resize(n);
    bool ok = get_host(f, e->h_creator.data(), sizeof(int32_t) * n) && get_host(f, e->h_head.data(), sizeof(int32_t) * M)
        && get_host(f, e->h_count.data(), sizeof(int32_t) * M) && get_host(f, e->h_height, sizeof(int32_t) * n)
        && get_host(f, e->h_seq, sizeof(int32_t) * n) && get_host(f, e->h_stale, (size_t)n)
        && get_dev(e, f, e->d_p0, sizeof(int32_t) * n, tmp) && get_dev(e, f, e->d_p1, sizeof(int32_t) * n, tmp)
        && get_dev(e, f, e->d_creator, sizeof(int32_t) * n, tmp) && get_dev(e, f, e->d_t, sizeof(double) * n, tmp)
        && get_dev(e, f, e->d_sig, (size_t)64 * n, tmp)
        && get_dev(e, f, e->d_row, sizeof(int32_t) * (size_t)nr * M, tmp)
        && get_dev(e, f, e->d_round, sizeof(int32_t) * nd, tmp) && get_dev(e, f, e->d_wit, (size_t)nd, tmp)
        && (e->wide ? get_dev(e, f, e->d_SMw, sizeof(unsigned) * (size_t)nd * e->NJ, tmp) : get_dev(e, f, e->d_SM, sizeof(u64) * nd, tmp))
        && get_dev(e, f, e->d_famous_ev, (size_t)n, tmp) && get_dev(e, f, e->d_idx, sizeof(int32_t) * n, tmp)
        && get_dev(e, f, e->d_tx, sizeof(int32_t) * H.n_tx, tmp)
        && get_dev(e, f, e->d_W, sizeof(int32_t) * RM, tmp) && get_dev(e, f, e->d_Wf, sizeof(int32_t) * RM, tmp)
        && get_dev(e, f, e->d_famous, RM, tmp) && get_dev(e, f, e->d_coin, RM, tmp)
        && (e->wide ? get_dev(e, f, e->d_Sw, sizeof(unsigned) * RM * e->NJ, tmp) : get_dev(e, f, e->d_S, sizeof(u64) * RM, tmp))
        && get_dev(e, f, e->d_consensus, (size_t)R, tmp)
        && get_dev(e, f, e->d_lastord, sizeof(int32_t) * M, tmp) && get_dev(e, f, e->d_cs_carry, sizeof(int32_t) * M, tmp)
        && get_dev(e, f, e->d_rbtot, sizeof(int32_t) * M, tmp) && get_dev(e, f, e->d_gchain, sizeof(int32_t) * (size_t)M * RB_RING, tmp)
        && get_dev(e, f, e->d_scal, sizeof(int32_t) * SC_COUNT, tmp);
    if (ok) {
        std::vector<uint8_t> idrec((size_t)36 * H.n_ids);
        ok = get_host(f, idrec.data(), idrec.size());
        for (size_t o = 0; ok && o < idrec.size(); o += 36) { Id32 k; int32_t v; memcpy(k.data(), &idrec[o], 32); memcpy(&v, &idrec[o + 32], 4); e->ids.emplace(k, v); }
    }
    fclose(f);
    if (!ok) { sw_destroy(e); return fail(nullptr, SW_E_ARG, "sw_load: %s is truncated or does not match its header", path); }
    // the derived columns live on the device too
    bool ok2 = cudaMemcpy(e->d_seq, e->h_seq, sizeof(int32_t) * n, cudaMemcpyHostToDevice) == cudaSuccess
        && cudaMemcpy(e->d_height, e->h_height, sizeof(int32_t) * n, cudaMemcpyHostToDevice) == cudaSuccess
        && cudaMemcpy(e->d_stale, e->h_stale, (size_t)n, cudaMemcpyHostToDevice) == cudaSuccess;
    if (!ok2) { sw_destroy(e); return fail(nullptr, SW_E_CUDA, "sw_load: device copy failed"); }
    e->n_events = n; e->n_divided = nd; e->n_tx = H.n_tx; e->n_rowed = nr; e->rb_epoch = H.rb_epoch;
    e->h_stale_cum.assign((size_t)n + 1, 0);
    for (int i = 0; i < n; i++) e->h_stale_cum[i + 1] = e->h_stale_cum[i] + e->h_stale[i];
    e->stats.events = n; e->stats.events_divided = nd;
    *out = e;
    return SW_OK;
}

// ---- several GPUs of one box: exchange buffers over NVLink peer memory (CUDA IPC, one process per GPU)
int sw_peer_handle(sw_engine *e, void *handle_out64) {
    if (!e || !handle_out64) return fail(e, SW_E_ARG, "bad argument");
    if (!e->wide) return fail(e, SW_E_UNSUPPORTED, "the M <= 64 path does not shard (replicas only): no peer exchange");
    CK(cudaSetDevice(e->device));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CK(cudaIpcGetMemHandle(&h, e->d_xbuf));
    memcpy(handle_out64, &h, 64);
    CK(cudaIpcGetMemHandle(&h, e->d_row));
    memcpy(reinterpret_cast<char *>(handle_out64) + 64, &h, 64);
    return SW_OK;
}

int sw_peer_connect(sw_engine *e, int rank, int nranks, const void *handles) {
    if (!e || !handles || nranks < 1 || nranks > 8 || rank < 0 || rank >= nranks) return fail(e, SW_E_ARG, "bad argument");
    if (!e->wide) return fail(e, SW_E_UNSUPPORTED, "the M <= 64 path does not shard (replicas only): no peer exchange");
    if (e->n_divided > 0) return fail(e, SW_E_ARG, "sw_peer_connect: connect before the first divide_rounds");
    CK(cudaSetDevice(e->device));
    for (int p = 0; p < nranks; p++) {
        if (p == rank) { e->x_peer[p] = e->d_xbuf; e->row_peer[p] = e->d_row; continue; }
        cudaIpcMemHandle_t h;
        memcpy(&h, reinterpret_cast<const char *>(handles) + (size_t)SW_PEER_HANDLE_BYTES * p, 64);
        void *ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        e->x_peer[p] = ptr;
        memcpy(&h, reinterpret_cast<const char *>(handles) + (size_t)SW_PEER_HANDLE_BYTES * p + 64, 64);
        ptr = nullptr;
        CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
        e->row_peer[p] = reinterpret_cast<int32_t *>(ptr);
    }
    // the ranks' barrier flag rows (128 bytes into the exchange buffer) as a device array
    unsigned *fl[8] = {nullptr};
    for (int p = 0; p < nranks; p++) fl[p] = reinterpret_cast<unsigned *>(reinterpret_cast<char *>(e->x_peer[p]) + 128);
    if (!e->d_xflags2) CK(cudaMalloc((void **)&e->d_xflags2, sizeof(unsigned *) * 8));
    CK(cudaMemcpy(e->d_xflags2, fl, sizeof fl, cudaMemcpyHostToDevice));
    e->rank = rank; e->nranks = nranks;
    return SW_OK;
}

}  // extern "C"
