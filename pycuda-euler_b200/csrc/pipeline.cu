// pipeline.cu -- the fused, device-resident hot path: encode -> canonical l-mer table ->
// vertex table -> ids -> D1-D6, plus the Euler tour / contig stage on the resident graph.
// Replaces eulercuda.constructDebruijnGraph (:183-264) + readLmersKmersCuda (:74-180) +
// findEulerTour (:407-436) with everything kept in HBM between stages.
#include "kernels.h"
#include "scan.cuh"
#include "sort.cuh"
#include "tmp.cuh"
#include "wide.cuh"
#include "bucket.cuh"
#include <stdlib.h>
#include <utility>

struct LtTable {
    DevBuf b;
    u64 cap = 0;
    int reserve(euler_ctx *ctx, u64 c)
    {
        EULER_TRY(dev_reserve(ctx, b, c * 12 + 256));
        cap = c;
        return EULER_OK;
    }
    u64 *keys() const { return (u64 *)b.p; }
    u32 *cnt() const { return (u32 *)((char *)b.p + cap * 8); }
    size_t bytes() const { return (size_t)cap * 12; }
};

// L2 residency hint for the table while the count kernel runs: table lines persist, everything else
// (the read stream) is treated as streaming.  Opt-in with EULER_B200_L2_PERSIST=1: on B200 the
// set-aside costs the other kernels more than the table gains (count 1.55 -> 1.65 ms, graph 1.7 -> 3.0 ms).
static void l2_window(euler_ctx *ctx, void *base, size_t bytes)
{
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("EULER_B200_L2_PERSIST");
        on = (e && atoi(e) == 1) ? 1 : 0;   // opt-in: see ctx.cu
    }
    if (!on || !ctx->persist_max || !ctx->window_max) return;
    cudaStreamAttrValue v;
    memset(&v, 0, sizeof(v));
    if (base && bytes) {
        const size_t nb = bytes < ctx->window_max ? bytes : ctx->window_max;
        v.accessPolicyWindow.base_ptr = base;
        v.accessPolicyWindow.num_bytes = nb;
        const double r = (double)ctx->persist_max / (double)nb;
        v.accessPolicyWindow.hitRatio = (float)(r > 1.0 ? 1.0 : r);
        v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
        v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    }
    cudaStreamSetAttribute(ctx->stream, cudaStreamAttributeAccessPolicyWindow, &v);
}

struct Pipeline {
    u32 l = 0, flags = 0;
    const void *d_buf = nullptr;
    const u64 *d_off = nullptr;
    u64 nreads = 0, n_bases = 0;
    // staged inputs of the host entry point
    DevArr<unsigned char> in_buf;
    DevArr<u64> in_off;
    DevArr<u32> start_bits;
    // canonical l-mer table (SoA) and canonical k-mer (vertex) table
    LtTable lt;  // keys u64[cap] followed by counts u32[cap] in ONE allocation (one L2 access-policy window covers both)
    DevArr<u32> lt_base, lt_eoff;
    DevArr<u64> lt_packed, side_keys;  // packed count table (packed.cu) and its wrap side table
    DevArr<u32> side_cnt;
    DevArr<unsigned char> lt_own;  // partitioned path: ownership bits per slot
    u64 lt_cap = 0;
    DevArr<u64> vt_keys;
    DevArr<u32> vt_id0, vt_id1;
    u64 vt_cap = 0;
    DevArr<u64> stats;  // [0] N_l [1] N_k [2] flags [3] U_l [4] V [5] E
    // graph artefacts
    DevArr<u64> lkeys, vkeys;
    DevArr<u32> lvals, loffs, ev1, ev2, lcount, ecount, lstart, estart;
    // table input (euler_pipeline_run_lmers): both-strand or canonical l-mers with counts instead of reads
    DevArr<u64> tbl_keys;
    DevArr<u32> tbl_cnt;
    u64 tbl_n = 0;
    bool from_table = false;
    DevArr<u64> lt_merged;  // merged count table (encode.cu, MERGED): 32-byte buckets {key, key, key, counters}
    DevArr<u32> vt_bbase;  // id of the first strand of each vertex-table bucket (slot-order ids)
    DevArr<u32> deg;  // paired degree regions u32[8 V] (common.cuh, DegOut) of the slot-order fast paths
    DevArr<euler_vertex> ev;
    DevArr<euler_edge> ee;
    DevArr<u32> lev, ent;
    // sort scratch (canonical ids)
    DevArr<u64> sort_k;
    DevArr<u32> sort_v, sort_hist;
    u64 U_l = 0, V = 0, E = 0;
    bool have_graph = false, expanded = false;
    // capacity memory: distinct canonical l-mers / k-mers seen on the last run of this input size
    u64 learned_bases = 0, learned_lc = 0, learned_vc = 0;
    u64 text_bytes = 0, text_n = 0, text_gen = 0;
    bool text_valid = false;  // contig text of the current graph is resident
    bool ingested = false;    // in_buf / in_off hold reads parsed on device by euler_ingest
    DevArr<u64> blk_keys, blk_cur;  // partitioned path, tables >> L2: keys regrouped by table region, run cursors
    void *recv_buf = nullptr;  // peer-visible receive buffer of the partitioned path (plain cudaMalloc)
    u64 recv_cap = 0;
    // 128-bit keys (l in 33..64, wide.cu): tables, high key words, first/last base codes per l-mer
    DevArr<K128> wlt_keys, wvt_keys;
    DevArr<u32> wlt_cnt;
    DevArr<u64> lkeys_hi, vkeys_hi;
    DevArr<unsigned char> tf;
    bool wide = false;
    // bucketed hot path (bucket.cuh): record regions, per-bucket cursors, look-back state, cross-bucket edge table
    DevBuf bk_records, bk_state;
    DevArr<u32> bk_cursors, bk_bvals, bk_perm, bk_newid, bk_tmp32a, bk_tmp32b, bk_tmp32c, bk_rows_a, bk_rows_b;
    DevArr<u64> bk_bkeys;
    DevArr<uint4 *> bk_dst;
    u32 bk_learned_rcap = 0, bk_learned_nb = 0;
    u64 bk_learned_bases = 0, bk_learned_u = 0, bk_learned_v = 0;
    u32 bk_learned_l = 0;
    void *bk_area[2] = {nullptr, nullptr};   // peer-visible bucket areas of the multi-GPU form (plain cudaMalloc)
    u64 bk_area_bytes[2] = {0, 0};
    u64 bk_dist_key = 0;
    u32 bk_dist_rcap = 0;
    u64 dist_bits_bases = ~0ull; u32 dist_bits_l = 0;   // what the read-start bitmap of the last euler_dist_count was built for
    u32 bk_dist_cap = 0;     // table capacity the last build of this geometry settled on
    DevArr<u32> bk_scursors;   // per-destination stream cursors of the multi-GPU form
    float bk_scatter_ms = 0;
    euler_stats st = {};
};

// the device buffers free themselves; only the IPC-exported allocations are raw
void pipeline_destroy(Pipeline *p)
{
    if (!p) return;
    if (p->recv_buf) cudaFree(p->recv_buf);
    for (int i = 0; i < 2; i++) if (p->bk_area[i]) cudaFree(p->bk_area[i]);
    delete p;
}

static u64 round_up(u64 x, u64 m) { return (x + m - 1) / m * m; }
// table capacity for `n` expected distinct keys at load factor ~0.55
static double table_load()
{
    static double lf = 0;
    if (lf == 0) {
        const char *e = getenv("EULER_B200_LOAD");
        lf = e ? atof(e) : 0.55;
        if (lf < 0.05 || lf > 0.95) lf = 0.55;
    }
    return lf;
}
// Minimizer-ordered homes (common.cuh) for tables that are big enough to matter; vertices are the
// shortest keys, so the minimizer length is bounded by k.  EULER_B200_MINHASH=0 turns it off.
static TableHash table_hash_for(u64 cap, u32 k)
{
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("EULER_B200_MINHASH");
        on = (e && atoi(e) != 0) ? 1 : 0;   // measured slower than the plain hash (bucket-load variance): opt-in
    }
    const u64 nb = cap / EULER_BUCKET;
    TableHash th = {0, 0};
    if (on && k >= 8 && nb > 64 * EULER_SPAN) {
        th.span_nb = (u32)(nb - EULER_SPAN);
        th.m = k < 12 ? k : 12;
    }
    return th;
}
// EULER_B200_PACKED=1 selects the packed quotient count table (packed.cu).  Measured on B200: it
// removes the DRAM misses (DRAM read 2.8 GB -> 0.26 GB per launch, L2 hit 55 % -> 71 %) but issues
// 56 % more instructions, and the kernel is issue/latency bound: 2.3 ms vs 1.5 ms.  Opt-in.
static bool use_packed_table()
{
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("EULER_B200_PACKED");
        on = (e && atoi(e) == 1) ? 1 : 0;
    }
    return on != 0;
}
// EULER_B200_BLOCK_MB: table size from which the partitioned path regroups keys for L2 (0 = never)
static u32 dist_block_min_mb()
{
    const char *e = getenv("EULER_B200_BLOCK_MB");
    return e ? (u32)atoi(e) : 512u;
}
// Co-hashed l-mer table (common.cuh).  Measured: on one GPU (config 2) the graph stage gains 0.15 ms and
// the count kernel loses 0.14 ms (12 more instructions per key) -- a wash, so it is off there; with a
// per-rank table far larger than L2 the graph stage gains 10 % (17.4 -> 15.6 ms on a 1 GB table), so the
// partitioned path turns it on together with the L2 blocking.  EULER_B200_COHASH=0/1 overrides both.
static bool use_cohash(bool dflt)
{
    const char *e = getenv("EULER_B200_COHASH");
    return e ? atoi(e) != 0 : dflt;
}
// EULER_B200_MERGED=1: count into the merged table (one sector per insert) and unpack it for the graph stage
static bool use_merged_table()
{
    const char *e = getenv("EULER_B200_MERGED");
    return e && atoi(e) == 1;
}
static u64 cap_for(u64 n) { return round_up((u64)((double)(n < 64 ? 64 : n) / table_load()) + 1, 1024); }

// ---- stages shared by the graph builds --------------------------------------------------------------------------------
// start of a build: the previous graph, its contig text and its stats are gone
static void begin_run(Pipeline *P, u32 l, u32 flags, bool wide, u64 nreads, u64 n_bases)
{
    P->l = l; P->flags = flags; P->wide = wide;
    P->have_graph = false; P->expanded = false; P->text_valid = false;
    memset(&P->st, 0, sizeof(P->st));
    P->st.n_reads = nreads; P->st.n_bases = n_bases;
}

// expected distinct canonical l-mers / k-mers of B bases of reads: the hint, else what the last run of this size
// counted, else B
static void estimate_from_reads(const Pipeline *P, u64 B, u64 hint, u64 &est_l, u64 &est_v)
{
    if (hint) { est_l = hint; est_v = hint + hint / 16; }
    else if (P->learned_bases == B && P->learned_lc) { est_l = P->learned_lc + P->learned_lc / 32; est_v = P->learned_vc + P->learned_vc / 32; }
    else { est_l = B ? B : 1; est_v = est_l; }
}

// table capacities for nkeys received keys: from the hint, else from what the last build of as many keys counted, else
// one l-mer per key
static void caps_from_keys(const Pipeline *P, u64 nkeys, u64 hint, u64 &lt_cap, u64 &vt_cap)
{
    const bool learned = !hint && P->learned_bases == nkeys && P->learned_lc;
    const u64 est = hint ? hint : (learned ? P->learned_lc : (nkeys ? nkeys : 1));
    lt_cap = cap_for(est); vt_cap = cap_for(learned ? P->learned_vc : est);
}

// the graph artefacts for ucap both-strand l-mers and vcap vertices; two-word keys add the high words and tf
static int reserve_graph(euler_ctx *ctx, Pipeline *P, u64 ucap, u64 vcap, bool wide)
{
    EULER_TRY(P->lkeys.reserve(ctx, ucap)); EULER_TRY(P->lvals.reserve(ctx, ucap)); EULER_TRY(P->loffs.reserve(ctx, ucap));
    EULER_TRY(P->ev1.reserve(ctx, ucap)); EULER_TRY(P->ev2.reserve(ctx, ucap));
    EULER_TRY(P->vkeys.reserve(ctx, vcap));
    EULER_TRY(P->lcount.reserve(ctx, 4 * vcap + 4)); EULER_TRY(P->ecount.reserve(ctx, 4 * vcap + 4));
    EULER_TRY(P->lstart.reserve(ctx, 4 * vcap + 4)); EULER_TRY(P->estart.reserve(ctx, 4 * vcap + 4));
    EULER_TRY(P->ev.reserve(ctx, vcap));
    if (wide) {
        EULER_TRY(P->lkeys_hi.reserve(ctx, ucap)); EULER_TRY(P->vkeys_hi.reserve(ctx, vcap));
        EULER_TRY(P->tf.reserve(ctx, ucap + 16));
    }
    return EULER_OK;
}

// zero what the edge kernels count degrees into: the paired regions (common.cuh, DegOut) or lcount / ecount
static int clear_degrees(euler_ctx *ctx, Pipeline *P, u64 V, bool paired)
{
    cudaStream_t s = ctx->stream;
    if (paired) {
        EULER_TRY(P->deg.reserve(ctx, 8 * V + 8));
        CUDA_TRY(ctx, cudaMemsetAsync(P->deg.ptr(), 0, (8 * V + 8) * sizeof(u32), s));
    } else {
        CUDA_TRY(ctx, cudaMemsetAsync(P->lcount.ptr(), 0, (4 * V + 4) * sizeof(u32), s));
        CUDA_TRY(ctx, cudaMemsetAsync(P->ecount.ptr(), 0, (4 * V + 4) * sizeof(u32), s));
    }
    return EULER_OK;
}

// EULER_RUN_EXPAND_EDGES: the per-edge arrays of the graph just built (two-word keys give their first bases in tf)
static int expand_edges(euler_ctx *ctx, Pipeline *P, u32 &launches)
{
    if (!(P->flags & EULER_RUN_EXPAND_EDGES)) return EULER_OK;
    const u64 E = P->E;
    launches += 1;
    EULER_TRY(P->ee.reserve(ctx, E)); EULER_TRY(P->lev.reserve(ctx, E)); EULER_TRY(P->ent.reserve(ctx, E));
    EULER_TRY(graph_setup_edges(ctx, P->wide ? nullptr : P->lkeys.ptr(), P->lvals.ptr(), P->loffs.ptr(), P->U_l, P->l, P->ev1.ptr(),
                                P->ev2.ptr(), P->lstart.ptr(), P->estart.ptr(), (u32)E, P->ee.ptr(), P->lev.ptr(), P->ent.ptr(),
                                P->wide ? P->tf.ptr() : nullptr));
    P->expanded = true;
    return EULER_OK;
}

// Tail of every build: wait for the graph and make it the current one, add its sizes, retries, launches and phase times
// to P->st (the driver has set its own fields) and copy that out.  ms_graph runs from ev[graph_from] to ev[graph_to].
// A build that counted (graph_from = 1) times the count ev[0] -> ev[1], the count kernel ev[4] -> ev[1] and ms_total
// over both; otherwise ms_total is the graph alone.  The per-bucket builds (path 1) time bkt_build ev[5] -> ev[2].
static int finish_run(euler_ctx *ctx, Pipeline *P, u64 lt_cap, u64 vt_cap, u32 retries, u32 launches, int graph_from, int graph_to,
                      euler_stats *stats)
{
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    P->have_graph = true;
    euler_stats &st = P->st;
    st.distinct_lmers = P->U_l; st.distinct_kmers = P->V; st.edge_count = P->E;
    st.lmer_table_capacity = lt_cap; st.kmer_table_capacity = vt_cap; st.retries = retries; st.kernel_launches = launches;
    cudaEventElapsedTime(&st.ms_graph, ctx->ev[graph_from], ctx->ev[graph_to]);
    if (graph_from == 1) {
        cudaEventElapsedTime(&st.ms_count, ctx->ev[0], ctx->ev[1]);
        cudaEventElapsedTime(&st.ms_total, ctx->ev[0], ctx->ev[graph_to]);
        cudaEventElapsedTime(&st.ms_count_kernel, ctx->ev[4], ctx->ev[1]);
    } else {
        st.ms_total = st.ms_graph;
    }
    if (st.path == 1) cudaEventElapsedTime(&st.ms_build_kernel, ctx->ev[5], ctx->ev[2]);
    if (stats) *stats = st;
    return EULER_OK;
}

// l in 33..64: the same stages over two-word keys (wide.cu).  Correctness-first: one thread per read,
// explicit both-strand l-mer arrays, ids in slot order or ascending (hi, lo) order.
static int pipeline_run_wide(euler_ctx *ctx, Pipeline *P, u32 l, u32 flags, u64 distinct_hint, euler_stats *stats)
{
    const u32 k = l - 1;
    const u64 B = P->n_bases;
    cudaStream_t s = ctx->stream;
    begin_run(P, l, flags, true, P->nreads, B);
    EULER_TRY(P->stats.reserve(ctx, 16));
    u64 est_l, est_v;
    estimate_from_reads(P, B, distinct_hint, est_l, est_v);
    u64 lt_cap = cap_for(est_l), vt_cap = cap_for(est_v);
    u64 h[8] = {0};
    u32 retries = 0, launches = 0;
    // EULER_B200_WIDE_TILED=0: the one-thread-per-read count kernel (needs a 16-byte aligned buffer otherwise)
    const char *wt = getenv("EULER_B200_WIDE_TILED");
    const bool wide_tiled = !(wt && atoi(wt) == 0) && (((uintptr_t)P->d_buf & 15) == 0);
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    if (wide_tiled) {
        EULER_TRY(P->start_bits.reserve(ctx, B / 32 + 2));
        P->dist_bits_bases = ~0ull;   // the bitmap no longer belongs to an euler_dist_count call
        EULER_TRY(enc_mark_starts(ctx, P->d_off, P->nreads, B, P->start_bits.ptr()));
        launches++;
    }
    while (true) {
        P->lt_cap = lt_cap; P->vt_cap = vt_cap;
        EULER_TRY(P->wlt_keys.reserve(ctx, lt_cap)); EULER_TRY(P->wlt_cnt.reserve(ctx, lt_cap)); EULER_TRY(P->lt_base.reserve(ctx, lt_cap));
        EULER_TRY(P->wvt_keys.reserve(ctx, vt_cap)); EULER_TRY(P->vt_id0.reserve(ctx, vt_cap));
        CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 16 * sizeof(u64), s));
        EULER_TRY(wide_table_clear(ctx, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), lt_cap));
        EULER_TRY(wide_table_clear(ctx, P->wvt_keys.ptr(), nullptr, vt_cap));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
        if (wide_tiled)
            EULER_TRY(wide_count_tiled(ctx, P->d_buf, B, P->start_bits.ptr(), l, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), lt_cap,
                                       P->stats.ptr()));
        else
            EULER_TRY(wide_count(ctx, P->d_buf, P->d_off, P->nreads, l, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), lt_cap, P->stats.ptr()));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
        EULER_TRY(wide_slot_scan(ctx, P->wlt_keys.ptr(), lt_cap, l, P->lt_base.ptr(), P->stats.ptr() + 3));
        EULER_TRY(wide_vertex_insert(ctx, P->wlt_keys.ptr(), lt_cap, l, P->wvt_keys.ptr(), vt_cap, P->stats.ptr() + 2));
        EULER_TRY(wide_slot_scan(ctx, P->wvt_keys.ptr(), vt_cap, k, P->vt_id0.ptr(), P->stats.ptr() + 4));
        launches += 4;
        EULER_TRY(read_u64s(ctx, P->stats.ptr(), h, 6));
        if ((h[2] & 3) == 0) break;
        if (++retries > 10) return euler_fail(ctx, EULER_ERR_OVERFLOW, "hash table overflow after %u regrows", retries);
        // The window counts are complete even when a table overflowed, and they bound the distinct counts: one regrow
        // is enough however small the hint or the learned size was (doubling alone gave up after 10 on large inputs).
        if (h[2] & 1) lt_cap = std::max(2 * lt_cap, cap_for(h[0]));
        if (h[2] & 2) vt_cap = std::max(2 * vt_cap, cap_for(h[1]));
    }
    const u64 N_l = h[0], N_k = h[1], U_l = h[3], V = h[4];
    const u64 E = 2 * N_l;
    P->U_l = U_l; P->V = V; P->E = E;
    if (V >= 0x3fffffffull || N_l >= 0x7fffffffull)
        return euler_fail(ctx, EULER_ERR_RANGE, "graph exceeds u32 ids (U_l=%llu V=%llu E=%llu)", U_l, V, E);
    EULER_TRY(reserve_graph(ctx, P, U_l, V, true));
    EULER_TRY(clear_degrees(ctx, P, V, false));
    EULER_TRY(wide_compact_vertices(ctx, P->wvt_keys.ptr(), P->vt_id0.ptr(), vt_cap, k, P->vkeys.ptr(), P->vkeys_hi.ptr()));
    EULER_TRY(wide_compact_lmers(ctx, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), P->lt_base.ptr(), lt_cap, l, P->lkeys.ptr(),
                                 P->lkeys_hi.ptr(), P->lvals.ptr()));
    const u32 *id1 = nullptr;
    if (flags & EULER_RUN_CANONICAL_IDS) {
        EULER_TRY(P->vt_id1.reserve(ctx, vt_cap));
        EULER_TRY(wide_sort(ctx, P->lkeys.ptr(), P->lkeys_hi.ptr(), P->lvals.ptr(), U_l, 2 * (int)l));
        EULER_TRY(wide_sort(ctx, P->vkeys.ptr(), P->vkeys_hi.ptr(), nullptr, V, 2 * (int)k));
        EULER_TRY(wide_assign_sorted_ids(ctx, P->vkeys.ptr(), P->vkeys_hi.ptr(), V, P->wvt_keys.ptr(), vt_cap, k, P->vt_id0.ptr(),
                                         P->vt_id1.ptr()));
        id1 = P->vt_id1.ptr();
        launches += 3 * ((2 * l + 7) / 8) + 3 * ((2 * k + 7) / 8) + 12;
    }
    EULER_TRY(wide_degree_slots(ctx, P->lkeys.ptr(), P->lkeys_hi.ptr(), P->lvals.ptr(), U_l, l, P->wvt_keys.ptr(), P->vt_id0.ptr(), id1,
                                vt_cap, P->lcount.ptr(), P->ecount.ptr(), P->ev1.ptr(), P->ev2.ptr(), P->tf.ptr()));
    EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lvals.ptr()}, U_l, P->loffs.ptr(), (u64 *)nullptr));
    EULER_TRY(graph_vertices_fused(ctx, P->lcount.ptr(), P->ecount.ptr(), P->vkeys.ptr(), V, P->lstart.ptr(), P->estart.ptr(),
                                   P->ev.ptr()));
    launches += 5;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], s));
    EULER_TRY(expand_edges(ctx, P, launches));
    P->learned_bases = B;
    P->learned_lc = (U_l + 1) / 2 + 16; P->learned_vc = (V + 1) / 2 + 16;
    P->st.n_kmer_windows = N_k; P->st.n_lmer_windows = N_l;
    return finish_run(ctx, P, lt_cap, vt_cap, retries, launches, 1, 2, stats);
}


// ---- the bucketed hot path (bucket.cuh): partition pass + per-bucket shared-memory build ------------------------------
// EULER_B200_BUCKETED=0 selects the round-1 global-table path below (also the fallback when a bucket does not fit
// its shared-memory table, e.g. one minimizer shared by a huge number of distinct k-mers).
static bool use_bucketed()
{
    const char *e = getenv("EULER_B200_BUCKETED");
    return !(e && atoi(e) == 0);
}
static u32 env_u32(const char *name, u32 dflt)
{
    const char *e = getenv(name);
    return e && atoi(e) > 0 ? (u32)atoi(e) : dflt;
}
static u64 pow2_at_least(u64 x)
{
    u64 p = 1;
    while (p < x) p <<= 1;
    return p;
}
#define EULER_FALLBACK 1   // internal: take the global-table path instead
#define BKT_MAX_DISTINCT 50000000ull   // distinct canonical l-mers up to which the bucketed path is taken by default

// One round of the per-bucket build over nb regions of rcap records, shared-memory tables of cap slots, ucap / vcap
// artefact entries and a boundary table of bcap: reserve all of it, let fill_regions() put the records in place (or
// only reset the stats words when they already are), build, and read the 8 stats words back into h.  The repair after
// a round is the driver's own.
template <typename Fill>
static int bkt_round(euler_ctx *ctx, Pipeline *P, u32 l, u32 nb, u32 rcap, u32 cap, u64 ucap, u64 vcap, u64 bcap, u32 &launches,
                     u64 *h, Fill fill_regions)
{
    EULER_TRY(dev_reserve(ctx, P->bk_records, (size_t)nb * rcap * 16 + 16));
    EULER_TRY(P->bk_cursors.reserve(ctx, nb));
    EULER_TRY(dev_reserve(ctx, P->bk_state, bkt_state_bytes(nb)));
    EULER_TRY(P->bk_bkeys.reserve(ctx, bcap)); EULER_TRY(P->bk_bvals.reserve(ctx, 2 * bcap));
    EULER_TRY(reserve_graph(ctx, P, ucap, vcap, false));
    EULER_TRY(fill_regions());
    BktBuild bb;
    bb.records = P->bk_records.p; bb.counts = P->bk_cursors.ptr(); bb.nb = nb; bb.nranks = 1; bb.rcap = rcap; bb.l = l; bb.cap = cap;
    bb.lkeys = P->lkeys.ptr(); bb.lvals = P->lvals.ptr(); bb.loffs = P->loffs.ptr(); bb.ev1 = P->ev1.ptr(); bb.ev2 = P->ev2.ptr(); bb.ucap = ucap;
    bb.vkeys = P->vkeys.ptr(); bb.lcount = P->lcount.ptr(); bb.ecount = P->ecount.ptr(); bb.lstart = P->lstart.ptr();
    bb.estart = P->estart.ptr(); bb.ev = P->ev.ptr(); bb.vcap = vcap;
    bb.state = P->bk_state.p; bb.bkeys = P->bk_bkeys.ptr(); bb.bvals = P->bk_bvals.ptr(); bb.bcap = bcap; bb.stats = P->stats.ptr();
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[5], ctx->stream));
    EULER_TRY(bkt_build(ctx, bb));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], ctx->stream));
    launches += 4;   // build, second pass, boundary publish, fix-up
    EULER_TRY(read_u64s(ctx, P->stats.ptr(), h, 8));   // the only host round trip of a steady-state step
    if (h[2] & BKT_FLAG_INTERNAL)
        return euler_fail(ctx, EULER_ERR_STATE, "internal: bucketed build consistency check failed (flags %llx)", h[2]);
    return EULER_OK;
}

static int pipeline_run_bucketed(euler_ctx *ctx, Pipeline *P, u32 l, u32 flags, u64 distinct_hint, euler_stats *stats)
{
    const u32 k = l - 1;
    const u64 B = P->n_bases;
    cudaStream_t s = ctx->stream;
    if (B >= (1ull << 40)) return EULER_FALLBACK;
    EULER_TRY(P->stats.reserve(ctx, 64));
    EULER_TRY(P->start_bits.reserve(ctx, B / 32 + 2));
    P->dist_bits_bases = ~0ull;   // the bitmap no longer belongs to an euler_dist_count call

    // geometry: buckets sized for a shared-memory table at ~45 % load
    const u32 cap = (env_u32("EULER_B200_BKT_CAP", 1536) + 255u) / 256u * 256u;   // 29 B per slot: 4 resident blocks per SM
    const bool learned = !distinct_hint && P->bk_learned_bases == B && P->bk_learned_l == l && P->bk_learned_nb;
    // a previous run of the same reads through the global-table path has left its distinct count as well
    const bool learned_gt = !distinct_hint && !learned && P->learned_bases == B && P->learned_lc;
    u64 est_c = distinct_hint ? distinct_hint : (learned ? (P->bk_learned_u + 1) / 2 : (learned_gt ? P->learned_lc : (B ? B : 1)));
    const char *le = getenv("EULER_B200_BKT_LOAD");
    const double per_bucket = (le && atof(le) > 0.05 && atof(le) < 0.9 ? atof(le) : 0.30) * (double)cap;   // mean table load (linear probing)
    u64 nb64 = learned ? P->bk_learned_nb : (u64)((double)est_c * 1.06 / per_bucket) + 1;
    // a hint that is far too small must not pile the whole input into a handful of buckets (every occurrence of every
    // l-mer would walk a full table before the repartition): at least one bucket per 128 Ki bases
    if (!learned && nb64 < (B >> 17)) nb64 = B >> 17;
    if (const u32 f = env_u32("EULER_B200_BKT_NB", 0)) nb64 = f;
    // Where the bucketed path pays: tables whose buckets stay few enough for the 12-mer minimizers to balance them and
    // for the scattered 16-byte record stores to stay inside the TLB reach (measured: 1.25e8 distinct l-mers -> 3.3e5
    // buckets with a 5x spread of the bucket sizes and a 59 GB record area).  Larger tables take the round-1 path
    // (global tables, L2-blocked); EULER_B200_BUCKETED=2 forces the bucketed path at any size.
    {
        const char *e = getenv("EULER_B200_BUCKETED");
        if (!(e && atoi(e) == 2) && est_c > BKT_MAX_DISTINCT) return EULER_FALLBACK;
    }
    if (nb64 > (1ull << 24)) return EULER_FALLBACK;
    u32 nb = (u32)nb64;
    // records: one per minimizer run cut at 16-base chunk boundaries, plus the orphans
    const u32 W = k - bk_m_of(k) + 1;
    const double rec_per_base = 2.0 / (W + 1.0) + 1.0 / 16.0 + 0.01;
    u32 rcap = learned && P->bk_learned_rcap ? P->bk_learned_rcap
                                            : (u32)((double)B * rec_per_base / nb * 1.5) + 64;
    // artefact capacities: known from a hint or the last run of this input, else a first build only counts
    u64 ucap = (distinct_hint || learned_gt) ? 2 * est_c + est_c / 4 + 1024 : (learned ? P->bk_learned_u + P->bk_learned_u / 64 + 1024 : 0);
    u64 vcap = (distinct_hint || learned_gt) ? 2 * est_c + est_c / 4 + 1024 : (learned ? P->bk_learned_v + P->bk_learned_v / 64 + 1024 : 0);
    u64 bcap = pow2_at_least((distinct_hint || learned || learned_gt ? est_c / 6 : est_c / 16) + 1024);

    u64 h[8] = {0};
    u32 retries = 0, launches = 0;
    bool need_part = true;
    EULER_TRY(P->bk_dst.reserve(ctx, 16));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    EULER_TRY(enc_mark_starts(ctx, P->d_off, P->nreads, B, P->start_bits.ptr()));
    launches++;
    while (true) {
        if ((u64)nb * rcap * 16 > (48ull << 30)) return EULER_FALLBACK;
        EULER_TRY(bkt_round(ctx, P, l, nb, rcap, cap, ucap, vcap, bcap, launches, h, [&]() -> int {
            if (!need_part) {
                CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr() + 2, 0, 6 * sizeof(u64), s));   // flags, totals, max region
                return EULER_OK;
            }
            uint4 *self = (uint4 *)P->bk_records.p;
            CUDA_TRY(ctx, cudaMemcpyAsync(P->bk_dst.ptr(), &self, sizeof(self), cudaMemcpyHostToDevice, s));
            CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 32 * sizeof(u64), s));
            CUDA_TRY(ctx, cudaMemsetAsync(P->bk_cursors.ptr(), 0, (size_t)nb * sizeof(u32), s));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
            EULER_TRY(bkt_partition(ctx, P->d_buf, B, P->start_bits.ptr(), l, 1, nb, 0, rcap, P->bk_dst.ptr(), P->bk_cursors.ptr(),
                                    P->stats.ptr()));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
            launches++;
            need_part = false;
            return EULER_OK;
        }));
        if (getenv("EULER_B200_BKT_TIMING")) {   // library built with -DBKT_TIMING: clock cycles per build phase, summed over the blocks
            u64 t[8];
            EULER_TRY(read_u64s(ctx, P->stats.ptr() + 16, t, 8));
            fprintf(stderr, "bkt_build phases (Mcycles over %u blocks): clear %.1f | A count %.1f | B vertices %.1f | C totals %.1f | D look-back %.1f | E1 vertex out %.1f | E2 edge out %.1f\n",
                    nb, t[0] / 1e6, t[1] / 1e6, t[2] / 1e6, t[3] / 1e6, t[4] / 1e6, t[5] / 1e6, t[6] / 1e6);
        }
        const u64 fl = h[2];
        if (!(fl & (BKT_FLAG_REGION | BKT_FLAG_TABLE | BKT_FLAG_OUTPUT | BKT_FLAG_BOUNDARY))) break;
        if (++retries > 8) return EULER_FALLBACK;
        if (fl & BKT_FLAG_REGION) {   // stats[6] = the largest region
            rcap = (u32)(h[6] + h[6] / 8 + 16);
            need_part = true;
        } else if (fl & BKT_FLAG_TABLE) {
            if (nb >= (1u << 22) || retries > 6) return EULER_FALLBACK;
            nb *= 4;   // far more distinct l-mers than estimated: partition again into more buckets
            rcap = rcap / 4 + rcap / 8 + 64;
            need_part = true;
        } else {
            if (fl & BKT_FLAG_OUTPUT) { ucap = h[3] + h[3] / 64 + 1024; vcap = h[4] + h[4] / 64 + 1024; }
            if (fl & BKT_FLAG_BOUNDARY) bcap *= 4;
        }
    }
    const u64 N_l = h[0], N_k = h[1], U_l = h[3], V = h[4], E = h[5];
    // u32 ids: vertices and distinct l-mers.  The edge total may pass 2^32 (E is exact, 64-bit): the compressed graph stays
    // exact and the `unsigned int` offsets of the reference layout (lmerOffsets, lstart / estart, EulerVertex.lp / .ep,
    // pydebruijn.py:90-101) are then kept modulo 2^32 -- they only address the expanded edge arrays, which need E < 2^32.
    if (V >= 0x3fffffffull || U_l >= 0xffffffffull)
        return euler_fail(ctx, EULER_ERR_RANGE, "graph exceeds u32 ids (U_l=%llu V=%llu E=%llu)", U_l, V, E);
    if ((flags & EULER_RUN_EXPAND_EDGES) && E >= 0xffffffffull)
        return euler_fail(ctx, EULER_ERR_RANGE, "expanded edges need E < 2^32 (E=%llu)", E);
    if (E != 2 * N_l) return euler_fail(ctx, EULER_ERR_STATE, "internal: edge total %llu != 2 N_l %llu", E, 2 * N_l);
    P->U_l = U_l; P->V = V; P->E = E;

    if (flags & EULER_RUN_CANONICAL_IDS) {
        // ids = rank in ascending key order (B14): sort the keys with their bucket-order index as payload, gather the rest
        const u64 nmax = U_l > V ? U_l : V;
        const u32 nblocks = (u32)((nmax + RS_TILE - 1) / RS_TILE);
        EULER_TRY(P->sort_k.reserve(ctx, nmax)); EULER_TRY(P->sort_v.reserve(ctx, nmax));
        EULER_TRY(P->sort_hist.reserve(ctx, (u64)256 * (nblocks ? nblocks : 1)));
        EULER_TRY(P->bk_perm.reserve(ctx, nmax)); EULER_TRY(P->bk_newid.reserve(ctx, V));
        EULER_TRY(P->bk_rows_a.reserve(ctx, 4 * V + 4)); EULER_TRY(P->bk_rows_b.reserve(ctx, 4 * V + 4));
        EULER_TRY(P->bk_tmp32a.reserve(ctx, U_l)); EULER_TRY(P->bk_tmp32b.reserve(ctx, U_l)); EULER_TRY(P->bk_tmp32c.reserve(ctx, U_l));
        EULER_TRY(bkt_iota(ctx, P->bk_perm.ptr(), V));
        EULER_TRY(radix_sort_pairs(ctx, P->vkeys.ptr(), P->bk_perm.ptr(), V, 2 * (int)k, P->sort_k.ptr(), P->sort_v.ptr(), P->sort_hist.ptr()));
        EULER_TRY(bkt_invert_perm(ctx, P->bk_perm.ptr(), V, P->bk_newid.ptr()));
        EULER_TRY(bkt_gather_rows(ctx, P->bk_perm.ptr(), V, P->lcount.ptr(), P->ecount.ptr(), P->bk_rows_a.ptr(), P->bk_rows_b.ptr()));
        std::swap(P->lcount, P->bk_rows_a);
        std::swap(P->ecount, P->bk_rows_b);
        EULER_TRY(bkt_iota(ctx, P->bk_perm.ptr(), U_l));
        EULER_TRY(radix_sort_pairs(ctx, P->lkeys.ptr(), P->bk_perm.ptr(), U_l, 2 * (int)l, P->sort_k.ptr(), P->sort_v.ptr(), P->sort_hist.ptr()));
        EULER_TRY(bkt_gather_edges(ctx, P->bk_perm.ptr(), U_l, P->bk_newid.ptr(), P->lvals.ptr(), P->ev1.ptr(), P->ev2.ptr(),
                                   P->bk_tmp32a.ptr(), P->bk_tmp32b.ptr(), P->bk_tmp32c.ptr()));
        std::swap(P->lvals, P->bk_tmp32a);
        std::swap(P->ev1, P->bk_tmp32b);
        std::swap(P->ev2, P->bk_tmp32c);
        EULER_TRY(P->loffs.reserve(ctx, U_l));
        EULER_TRY(P->lstart.reserve(ctx, 4 * V + 4)); EULER_TRY(P->estart.reserve(ctx, 4 * V + 4)); EULER_TRY(P->ev.reserve(ctx, V));
        EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lvals.ptr()}, U_l, P->loffs.ptr(), (u64 *)nullptr));
        EULER_TRY(graph_vertices_fused(ctx, P->lcount.ptr(), P->ecount.ptr(), P->vkeys.ptr(), V, P->lstart.ptr(), P->estart.ptr(), P->ev.ptr()));
        launches += 3 * ((2 * l + 7) / 8) + 3 * ((2 * k + 7) / 8) + 8;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[6], s));
    EULER_TRY(expand_edges(ctx, P, launches));
    P->learned_bases = B;
    P->learned_lc = (U_l + 1) / 2 + 16; P->learned_vc = (V + 1) / 2 + 16;
    P->bk_learned_bases = B; P->bk_learned_l = l; P->bk_learned_nb = nb; P->bk_learned_u = U_l; P->bk_learned_v = V;
    P->bk_learned_rcap = (u32)(h[6] + h[6] / 8 + 16);
    // a hint that was far off: size the buckets from what was counted
    {
        const u64 want = (u64)((double)((U_l + 1) / 2) * 1.06 / per_bucket) + 1;
        if (!env_u32("EULER_B200_BKT_NB", 0) && (want * 2 < nb || want > (u64)nb * 2)) { P->bk_learned_nb = (u32)want; P->bk_learned_rcap = 0; }
    }
    euler_stats &st = P->st;
    st.n_kmer_windows = N_k; st.n_lmer_windows = N_l;
    st.path = 1; st.n_buckets = nb; st.bucket_records = h[6]; st.redo_buckets = (u32)h[7];
    return finish_run(ctx, P, (u64)nb * cap, (u64)nb * cap, retries, launches, 1, 6, stats);
}

static int pipeline_run(euler_ctx *ctx, Pipeline *P, u32 l, u32 flags, u64 distinct_hint, euler_stats *stats)
{
    if (l < 2 || l > 64) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,64]", l);
    if (l > 32) return pipeline_run_wide(ctx, P, l, flags, distinct_hint, stats);
    const u32 k = l - 1;
    const u64 B = P->n_bases;
    cudaStream_t s = ctx->stream;
    begin_run(P, l, flags, false, P->nreads, B);
    if (!P->from_table && use_bucketed()) {   // it changes nothing of P->st or the graph state before it falls back
        const int rc = pipeline_run_bucketed(ctx, P, l, flags, distinct_hint, stats);
        if (rc != EULER_FALLBACK) return rc;
    }

    EULER_TRY(P->stats.reserve(ctx, 16));
    EULER_TRY(P->start_bits.reserve(ctx, B / 32 + 2));
    P->dist_bits_bases = ~0ull;   // the bitmap no longer belongs to an euler_dist_count call

    u64 est_l, est_v;
    estimate_from_reads(P, B, distinct_hint, est_l, est_v);
    const bool from_table = P->from_table;
    if (from_table && !distinct_hint) { est_l = P->tbl_n ? P->tbl_n : 1; est_v = 2 * est_l; }
    u64 lt_cap = cap_for(est_l), vt_cap = cap_for(est_v);
    // packed count table: power-of-two bucket count, load factor in (0.375, 0.75]
    bool packed = !from_table && use_packed_table();
    bool merged = !from_table && !packed && use_merged_table() && !table_hash_for(lt_cap, k).span_nb;
    if (merged) lt_cap = round_up(lt_cap / 3 * 4 + 4, 1024);   // three key slots per 4-word bucket
    u32 pk_b = 8;
    const u64 side_cap = 16384;
    if (packed) {
        while (((u64)EULER_BUCKET << pk_b) * 3 < est_l * 4 && pk_b < 31) pk_b++;
        lt_cap = (u64)EULER_BUCKET << pk_b;
    }

    u64 h[8] = {0};
    TableHash lth = {0, 0}, vth = {0, 0};
    u32 retries = 0, launches = 1;  // mark_starts
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    if (!from_table) EULER_TRY(enc_mark_starts(ctx, P->d_off, P->nreads, B, P->start_bits.ptr()));
    while (true) {
        P->lt_cap = lt_cap; P->vt_cap = vt_cap;
        EULER_TRY(P->lt.reserve(ctx, lt_cap));
        EULER_TRY(P->lt_base.reserve(ctx, lt_cap));
        EULER_TRY(P->lt_eoff.reserve(ctx, lt_cap));
        EULER_TRY(P->vt_keys.reserve(ctx, vt_cap));
        EULER_TRY(P->vt_id0.reserve(ctx, vt_cap));
        CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 16 * sizeof(u64), s));
        EULER_TRY(graph_table_clear(ctx, P->vt_keys.ptr(), nullptr, vt_cap));
        vth = table_hash_for(vt_cap, k);
        if (packed) {
            EULER_TRY(P->lt_packed.reserve(ctx, lt_cap));
            EULER_TRY(P->side_keys.reserve(ctx, side_cap)); EULER_TRY(P->side_cnt.reserve(ctx, side_cap));
            CUDA_TRY(ctx, cudaMemsetAsync(P->lt_packed.ptr(), 0, lt_cap * sizeof(u64), s));
            EULER_TRY(graph_table_clear(ctx, P->side_keys.ptr(), P->side_cnt.ptr(), side_cap));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
            EULER_TRY(enc_count_packed(ctx, P->d_buf, B, P->start_bits.ptr(), l, P->lt_packed.ptr(), pk_b, P->side_keys.ptr(),
                                       P->side_cnt.ptr(), side_cap, P->stats.ptr()));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
            EULER_TRY(enc_unpack(ctx, P->lt_packed.ptr(), pk_b, P->side_keys.ptr(), P->side_cnt.ptr(), side_cap,
                                 P->stats.ptr() + 7, P->lt.keys(), P->lt.cnt()));
            launches += 2;
        } else if (from_table) {
            // the table of a previous count (e.g. the per-rank tables of the partitioned path, joined): canonical insert,
            // both-strand count v -> canonical count (v for a palindrome is 2n)
            EULER_TRY(graph_table_clear(ctx, P->lt.keys(), P->lt.cnt(), lt_cap));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
            EULER_TRY(unitig_dict_table(ctx, P->tbl_keys.ptr(), P->tbl_cnt.ptr(), P->tbl_n, l, P->lt.keys(), P->lt.cnt(), lt_cap,
                                        P->stats.ptr() + 2));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
        } else if (merged) {
            EULER_TRY(P->lt_merged.reserve(ctx, lt_cap));
            EULER_TRY(enc_merged_clear(ctx, P->lt_merged.ptr(), lt_cap));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
            EULER_TRY(enc_count_merged(ctx, P->d_buf, B, P->start_bits.ptr(), l, P->lt_merged.ptr(), lt_cap, use_cohash(false),
                                       P->stats.ptr()));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
            EULER_TRY(enc_merged_unpack(ctx, P->lt_merged.ptr(), lt_cap, P->lt.keys(), P->lt.cnt()));
            launches += 2;
        } else {
            EULER_TRY(graph_table_clear(ctx, P->lt.keys(), P->lt.cnt(), lt_cap));
            l2_window(ctx, P->lt.b.p, P->lt.bytes());
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
            lth = table_hash_for(lt_cap, k);
            if (!lth.span_nb && use_cohash(false)) lth.m = EULER_PREFIX_HOME;
            EULER_TRY(enc_count_canonical(ctx, P->d_buf, B, P->start_bits.ptr(), l, P->lt.keys(), P->lt.cnt(), lt_cap,
                                          lth, P->stats.ptr()));
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
            l2_window(ctx, nullptr, 0);
        }
        launches += 4;  // count, l-mer pair scan, vertex insert, vertex slot scan
        EULER_TRY(graph_lt_scan(ctx, P->lt.keys(), P->lt.cnt(), lt_cap, l, P->lt_base.ptr(), P->lt_eoff.ptr(),
                                P->stats.ptr() + 3));
        EULER_TRY(graph_vertex_insert(ctx, P->lt.keys(), lt_cap, l, P->vt_keys.ptr(), vt_cap, vth, P->stats.ptr() + 2));
        EULER_TRY(graph_slot_scan(ctx, P->vt_keys.ptr(), vt_cap, k, P->vt_id0.ptr(), P->stats.ptr() + 4));
        EULER_TRY(read_u64s(ctx, P->stats.ptr(), h, 6));
        if (merged && (h[2] & 7) == 0 && (h[3] >> 32) != 2 * h[0]) {
            // a 16-bit counter of the merged table overflowed: redo with the SoA table and its 32-bit counters
            merged = false;
            lt_cap = lt_cap / 4 * 3;
            retries++;
            continue;
        }
        if ((h[2] & 7) == 0) break;
        if (++retries > 10) return euler_fail(ctx, EULER_ERR_OVERFLOW, "hash table overflow after %u regrows", retries);
        if (h[2] & 4) packed = false;   // wrap side table full (extreme repeats): use the SoA kernel
        if (h[2] & 1) { lt_cap *= 2; pk_b++; }
        if (h[2] & 2) vt_cap *= 2;
    }
    const u64 N_l = from_table ? (h[3] >> 32) / 2 : h[0], N_k = h[1], U_l = h[3] & 0xffffffffull, V = h[4];
    const u64 E = 2 * N_l;
    P->U_l = U_l; P->V = V; P->E = E;
    if (V >= 0x3fffffffull || N_l >= 0x7fffffffull)
        return euler_fail(ctx, EULER_ERR_RANGE, "graph exceeds u32 ids (U_l=%llu V=%llu E=%llu)", U_l, V, E);
    if ((h[3] >> 32) != E) return euler_fail(ctx, EULER_ERR_STATE, "internal: edge total %llu != 2 N_l %llu", h[3] >> 32, E);

    EULER_TRY(reserve_graph(ctx, P, U_l, V, false));
    const bool paired = !(flags & EULER_RUN_CANONICAL_IDS);   // slot-order ids: the strands of a vertex have adjacent ids
    EULER_TRY(clear_degrees(ctx, P, V, paired));
    EULER_TRY(graph_compact_vertices(ctx, P->vt_keys.ptr(), P->vt_id0.ptr(), vt_cap, k, P->vkeys.ptr()));
    VertexTable vt = {P->vt_keys.ptr(), P->vt_id0.ptr(), nullptr, vt_cap, k, vth};
    if (flags & EULER_RUN_CANONICAL_IDS) {
        // ids = rank in ascending key order (B14): sort both-strand l-mers and vertices, then D1 over the arrays
        const u64 nmax = U_l > V ? U_l : V;
        const u32 nblocks = (u32)((nmax + RS_TILE - 1) / RS_TILE);
        EULER_TRY(P->sort_k.reserve(ctx, nmax)); EULER_TRY(P->sort_v.reserve(ctx, nmax));
        EULER_TRY(P->sort_hist.reserve(ctx, (u64)256 * nblocks));
        EULER_TRY(P->vt_id1.reserve(ctx, vt_cap));
        EULER_TRY(graph_compact_lmers(ctx, P->lt.keys(), P->lt.cnt(), P->lt_base.ptr(), lt_cap, l, P->lkeys.ptr(),
                                      P->lvals.ptr()));
        EULER_TRY(radix_sort_pairs(ctx, P->lkeys.ptr(), P->lvals.ptr(), U_l, 2 * (int)l, P->sort_k.ptr(), P->sort_v.ptr(),
                                   P->sort_hist.ptr()));
        EULER_TRY(radix_sort_pairs(ctx, P->vkeys.ptr(), nullptr, V, 2 * (int)k, P->sort_k.ptr(), nullptr, P->sort_hist.ptr()));
        EULER_TRY(graph_assign_sorted_ids(ctx, P->vkeys.ptr(), V, P->vt_keys.ptr(), vt_cap, k, vth, P->vt_id0.ptr(),
                                          P->vt_id1.ptr()));
        vt.id1 = P->vt_id1.ptr();
        EULER_TRY(graph_degree_slots(ctx, P->lkeys.ptr(), P->lvals.ptr(), U_l, l, vt, P->lcount.ptr(), P->ecount.ptr(),
                                     P->ev1.ptr(), P->ev2.ptr()));
        EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lvals.ptr()}, U_l, P->loffs.ptr(), (u64 *)nullptr));
        launches += 3 * ((2 * l + 7) / 8) + 3 * ((2 * k + 7) / 8) + 5;
    } else {
        // fast path: ids in table-slot order, one fused pass over the l-mer table
        EULER_TRY(P->vt_bbase.reserve(ctx, vt_cap / EULER_BUCKET + 1));
        EULER_TRY(graph_bucket_bases(ctx, P->vt_id0.ptr(), vt_cap, P->vt_bbase.ptr()));
        vt.bbase = P->vt_bbase.ptr();
        EULER_TRY(graph_edges_fused(ctx, P->lt.keys(), P->lt.cnt(), P->lt_base.ptr(), P->lt_eoff.ptr(), lt_cap, l, vt,
                                    P->lkeys.ptr(), P->lvals.ptr(), P->loffs.ptr(), P->ev1.ptr(), P->ev2.ptr(),
                                    P->lcount.ptr(), P->ecount.ptr(), P->deg.ptr()));
        launches += 3;   // compact_vertices, bucket_bases, edges_fused
    }
    // scans of the degree slots + EulerVertex records in one pass
    if (paired)
        EULER_TRY(graph_vertices_paired(ctx, P->deg.ptr(), k, P->vkeys.ptr(), V, P->lcount.ptr(), P->ecount.ptr(), P->lstart.ptr(),
                                        P->estart.ptr(), P->ev.ptr()));
    else
        EULER_TRY(graph_vertices_fused(ctx, P->lcount.ptr(), P->ecount.ptr(), P->vkeys.ptr(), V, P->lstart.ptr(), P->estart.ptr(),
                                       P->ev.ptr()));
    launches += 1;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], s));
    EULER_TRY(expand_edges(ctx, P, launches));
    P->learned_bases = B;
    // canonical distinct counts: palindromes are rare, U/2 rounded up is a safe learned size
    P->learned_lc = (U_l + 1) / 2 + 16; P->learned_vc = (V + 1) / 2 + 16;
    P->st.n_kmer_windows = N_k; P->st.n_lmer_windows = N_l;
    return finish_run(ctx, P, lt_cap, vt_cap, retries, launches, 1, 2, stats);
}

// per-rank build of the partitioned path over 16-byte keys (wide_dist.cu); same contract as dist_build_impl
static int wide_dist_build_impl(euler_ctx *ctx, Pipeline *P, const void *d_keys, uint64_t nkeys, uint32_t nregions,
                                uint64_t region_stride, const uint64_t *region_counts, uint32_t l, uint32_t rank, uint32_t nranks,
                                uint64_t distinct_hint, euler_stats *stats)
{
    if (nranks > 8) return euler_fail(ctx, EULER_ERR_ARG, "128-bit keys: at most 8 ranks");
    cudaStream_t s = ctx->stream;
    const u32 k = l - 1;
    begin_run(P, l, 0, true, 0, 0);
    EULER_TRY(P->stats.reserve(ctx, 64));
    u64 lt_cap, vt_cap;
    caps_from_keys(P, nkeys, distinct_hint, lt_cap, vt_cap);
    u64 h[8] = {0};
    u32 retries = 0, launches = 0;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    while (true) {
        P->lt_cap = lt_cap; P->vt_cap = vt_cap;
        EULER_TRY(P->wlt_keys.reserve(ctx, lt_cap)); EULER_TRY(P->wlt_cnt.reserve(ctx, lt_cap)); EULER_TRY(P->lt_base.reserve(ctx, lt_cap));
        EULER_TRY(P->lt_own.reserve(ctx, lt_cap));
        EULER_TRY(P->wvt_keys.reserve(ctx, vt_cap)); EULER_TRY(P->vt_id0.reserve(ctx, vt_cap));
        CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 8 * sizeof(u64), s));
        EULER_TRY(wide_table_clear(ctx, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), lt_cap));
        EULER_TRY(wide_table_clear(ctx, P->wvt_keys.ptr(), nullptr, vt_cap));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
        for (u32 r = 0; r < nregions; r++)
            EULER_TRY(wide_count_keys(ctx, (const K128 *)d_keys + (u64)r * region_stride, region_counts[r], P->wlt_keys.ptr(),
                                      P->wlt_cnt.ptr(), lt_cap, P->stats.ptr()));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
        EULER_TRY(wide_own_flags(ctx, P->wlt_keys.ptr(), lt_cap, l, rank, nranks, P->lt_own.ptr()));
        EULER_TRY(wide_homed_scan(ctx, P->wlt_keys.ptr(), P->lt_own.ptr(), lt_cap, l, P->lt_base.ptr(), P->stats.ptr() + 3));
        EULER_TRY(wide_dist_vertex_insert(ctx, P->wlt_keys.ptr(), lt_cap, l, P->lt_own.ptr(), P->wvt_keys.ptr(), vt_cap,
                                          P->stats.ptr() + 2));
        EULER_TRY(wide_slot_scan(ctx, P->wvt_keys.ptr(), vt_cap, k, P->vt_id0.ptr(), P->stats.ptr() + 4));
        launches += nregions + 4;
        EULER_TRY(read_u64s(ctx, P->stats.ptr(), h, 6));
        if ((h[2] & 3) == 0) break;
        if (++retries > 8) return euler_fail(ctx, EULER_ERR_OVERFLOW, "hash table overflow after %u regrows", retries);
        if (h[2] & 1) lt_cap *= 2;
        if (h[2] & 2) vt_cap *= 2;
    }
    const u64 U_l = h[3], V = h[4];
    P->U_l = U_l; P->V = V;
    if (V >= 0x3fffffffull || U_l >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "graph exceeds u32 ids");
    EULER_TRY(reserve_graph(ctx, P, U_l, V, true));
    EULER_TRY(clear_degrees(ctx, P, V, false));
    EULER_TRY(wide_compact_vertices(ctx, P->wvt_keys.ptr(), P->vt_id0.ptr(), vt_cap, k, P->vkeys.ptr(), P->vkeys_hi.ptr()));
    EULER_TRY(wide_compact_homed(ctx, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), P->lt_own.ptr(), P->lt_base.ptr(), lt_cap, l,
                                 P->lkeys.ptr(), P->lkeys_hi.ptr(), P->lvals.ptr()));
    EULER_TRY(wide_degree_slots(ctx, P->lkeys.ptr(), P->lkeys_hi.ptr(), P->lvals.ptr(), U_l, l, P->wvt_keys.ptr(), P->vt_id0.ptr(),
                                nullptr, vt_cap, P->lcount.ptr(), P->ecount.ptr(), P->ev1.ptr(), P->ev2.ptr(), P->tf.ptr()));
    EULER_TRY(wide_foreign_in_edges(ctx, P->wlt_keys.ptr(), P->wlt_cnt.ptr(), P->lt_own.ptr(), lt_cap, l, P->wvt_keys.ptr(),
                                    P->vt_id0.ptr(), vt_cap, P->ecount.ptr()));
    // offsets modulo 2^32 and the exact 64-bit edge total, as in dist_build_impl's large path
    EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lvals.ptr()}, U_l, P->loffs.ptr(), (u64 *)nullptr));
    EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lcount.ptr()}, 4 * V, P->lstart.ptr(), (u64 *)nullptr));
    EULER_TRY(scan_exclusive(ctx, ScanInU32{P->ecount.ptr()}, 4 * V, P->estart.ptr(), (u64 *)nullptr));
    EULER_TRY(graph_setup_vertices(ctx, P->vkeys.ptr(), V, P->lcount.ptr(), P->lstart.ptr(), P->ecount.ptr(), P->estart.ptr(),
                                   P->ev.ptr()));
    EULER_TRY(graph_sum_u32(ctx, P->lvals.ptr(), U_l, P->stats.ptr() + 6));
    u64 E = 0;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], s));
    EULER_TRY(read_u64(ctx, P->stats.ptr() + 6, &E));
    launches += 10;
    P->E = E;
    P->learned_bases = nkeys;
    P->learned_lc = h[5] + h[5] / 32 + 16;
    P->learned_vc = (V + 1) / 2 + V / 32 + 16;
    P->st.n_lmer_windows = nkeys;
    return finish_run(ctx, P, lt_cap, vt_cap, retries, launches, 1, 2, stats);
}

static Pipeline *get_pipe(euler_ctx *ctx)
{
    if (!ctx->pipe) ctx->pipe = new Pipeline();
    return ctx->pipe;
}

extern "C" {

int euler_pipeline_run_dev(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                           uint32_t l, uint32_t flags, uint64_t distinct_hint, euler_stats *stats)
{
    if (!ctx) return EULER_ERR_ARG;
    if ((!d_buf && n_bases) || !d_read_off) return euler_fail(ctx, EULER_ERR_ARG, "null device input");
    if (((uintptr_t)d_buf & 15) != 0) return euler_fail(ctx, EULER_ERR_ARG, "d_buf must be 16-byte aligned");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    P->d_buf = d_buf; P->d_off = (const u64 *)d_read_off; P->nreads = nreads; P->n_bases = n_bases;
    return pipeline_run(ctx, P, l, flags, distinct_hint, stats);
}

int euler_pipeline_run_host(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t l,
                            uint32_t flags, uint64_t distinct_hint, euler_stats *stats)
{
    if (!ctx) return EULER_ERR_ARG;
    if (!read_off) return euler_fail(ctx, EULER_ERR_ARG, "null read_off");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    const u64 B = read_off[nreads];
    if (B && !buf) return euler_fail(ctx, EULER_ERR_ARG, "null buf");
    P->ingested = false;
    EULER_TRY(P->in_buf.reserve(ctx, B + 16));
    EULER_TRY(P->in_off.reserve(ctx, nreads + 1));
    if (B) CUDA_TRY(ctx, cudaMemcpyAsync(P->in_buf.ptr(), buf, B, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(P->in_off.ptr(), read_off, (nreads + 1) * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    P->d_buf = P->in_buf.ptr(); P->d_off = P->in_off.ptr(); P->nreads = nreads; P->n_bases = B;
    return pipeline_run(ctx, P, l, flags, distinct_hint, stats);
}

// graph stage on a given l-mer table (keys: either strand or both, counts: both-strand counts); l <= 32
int euler_pipeline_run_lmers(euler_ctx *ctx, const uint64_t *keys, const uint32_t *counts, uint64_t n, uint32_t l, uint32_t flags,
                             euler_stats *stats)
{
    if (!ctx) return EULER_ERR_ARG;
    if (n && (!keys || !counts)) return euler_fail(ctx, EULER_ERR_ARG, "null table");
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,32]", l);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    P->ingested = false;
    EULER_TRY(P->tbl_keys.reserve(ctx, n + 1));
    EULER_TRY(P->tbl_cnt.reserve(ctx, n + 1));
    if (n) {
        CUDA_TRY(ctx, cudaMemcpyAsync(P->tbl_keys.ptr(), keys, n * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
        CUDA_TRY(ctx, cudaMemcpyAsync(P->tbl_cnt.ptr(), counts, n * sizeof(u32), cudaMemcpyHostToDevice, ctx->stream));
    }
    P->tbl_n = n; P->from_table = true;
    P->d_buf = nullptr; P->d_off = nullptr; P->nreads = 0; P->n_bases = 0;
    const int rc = pipeline_run(ctx, P, l, flags, 0, stats);
    P->from_table = false;
    return rc;
}

static int artifact(euler_ctx *ctx, int which, void **p, u64 *bytes)
{
    Pipeline *P = ctx->pipe;
    if (!P || !P->have_graph) return euler_fail(ctx, EULER_ERR_STATE, "no pipeline run to read from");
    const u64 U = P->U_l, V = P->V, E = P->E;
    switch (which) {
    case EULER_ART_LMER_KEYS: *p = P->lkeys.ptr(); *bytes = U * 8; break;
    case EULER_ART_LMER_VALUES: *p = P->lvals.ptr(); *bytes = U * 4; break;
    case EULER_ART_LMER_OFFSETS: *p = P->loffs.ptr(); *bytes = U * 4; break;
    case EULER_ART_KMER_KEYS: *p = P->vkeys.ptr(); *bytes = V * 8; break;
    case EULER_ART_LMER_KEYS_HI:
    case EULER_ART_KMER_KEYS_HI:
        if (!P->wide) return euler_fail(ctx, EULER_ERR_STATE, "high key words exist only for l > 32");
        if (which == EULER_ART_LMER_KEYS_HI) { *p = P->lkeys_hi.ptr(); *bytes = U * 8; }
        else { *p = P->vkeys_hi.ptr(); *bytes = V * 8; }
        break;
    case EULER_ART_LCOUNT: *p = P->lcount.ptr(); *bytes = 4 * V * 4; break;
    case EULER_ART_ECOUNT: *p = P->ecount.ptr(); *bytes = 4 * V * 4; break;
    case EULER_ART_LSTART: *p = P->lstart.ptr(); *bytes = 4 * V * 4; break;
    case EULER_ART_ESTART: *p = P->estart.ptr(); *bytes = 4 * V * 4; break;
    case EULER_ART_EV: *p = P->ev.ptr(); *bytes = V * sizeof(euler_vertex); break;
    case EULER_ART_EDGE_V1: *p = P->ev1.ptr(); *bytes = U * 4; break;
    case EULER_ART_EDGE_V2: *p = P->ev2.ptr(); *bytes = U * 4; break;
    case EULER_ART_EE:
    case EULER_ART_LEV:
    case EULER_ART_ENT:
        if (!P->expanded) return euler_fail(ctx, EULER_ERR_STATE, "edges were not expanded (EULER_RUN_EXPAND_EDGES)");
        if (which == EULER_ART_EE) { *p = P->ee.ptr(); *bytes = E * sizeof(euler_edge); }
        else if (which == EULER_ART_LEV) { *p = P->lev.ptr(); *bytes = E * 4; }
        else { *p = P->ent.ptr(); *bytes = E * 4; }
        break;
    default: return euler_fail(ctx, EULER_ERR_ARG, "unknown artefact %d", which);
    }
    return EULER_OK;
}

int euler_pipeline_artifact_bytes(euler_ctx *ctx, int which, uint64_t *bytes)
{
    if (!ctx || !bytes) return EULER_ERR_ARG;
    void *p; u64 b;
    EULER_TRY(artifact(ctx, which, &p, &b));
    *bytes = b;
    return EULER_OK;
}

int euler_pipeline_download(euler_ctx *ctx, int which, void *host_dst, uint64_t cap_bytes)
{
    if (!ctx) return EULER_ERR_ARG;
    void *p; u64 b;
    EULER_TRY(artifact(ctx, which, &p, &b));
    if (b > cap_bytes) return euler_fail(ctx, EULER_ERR_ARG, "destination too small (%llu > %llu)", b, (u64)cap_bytes);
    if (b) {
        if (!host_dst) return euler_fail(ctx, EULER_ERR_ARG, "null destination");
        CUDA_TRY(ctx, cudaMemcpyAsync(host_dst, p, b, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return EULER_OK;
}

int euler_pipeline_device_ptr(euler_ctx *ctx, int which, void **dptr)
{
    if (!ctx || !dptr) return EULER_ERR_ARG;
    u64 b;
    return artifact(ctx, which, dptr, &b);
}

// findEulerTour eulercuda.py:407-436 + findEulerDevice pyeulertour.py:715-793 on the resident graph
int euler_pipeline_contigs(euler_ctx *ctx, char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    if (!ctx || !out_bytes || !ncontigs) return EULER_ERR_ARG;
    Pipeline *P = ctx->pipe;
    if (!P || !P->have_graph || !P->expanded)
        return euler_fail(ctx, EULER_ERR_STATE, "contigs need a pipeline run with EULER_RUN_EXPAND_EDGES");
    const u32 E = (u32)P->E, V = (u32)P->V;
    *ncontigs = 0;
    if (!E) { *out_bytes = 0; return EULER_OK; }
    if (!out || !P->text_valid || P->text_gen != ctx->text_gen) {  // sizing call, first call, or another emission overwrote the shared text buffer: run the tour now
        DevTmp<euler_succ_vertex> sv(ctx, E);
        DevTmp<u32> D(ctx, E), C(ctx, E), cmap(ctx, E), mark(ctx, E);
        DevTmp<u64> cnt(ctx, 1);
        TMP_CHECK(ctx, sv); TMP_CHECK(ctx, D); TMP_CHECK(ctx, C); TMP_CHECK(ctx, cmap); TMP_CHECK(ctx, mark); TMP_CHECK(ctx, cnt);
        EULER_TRY(tour_reset_successors(ctx, P->ee.ptr(), E));  // idempotent across repeated calls
        EULER_TRY(tour_assign_successor(ctx, P->ev.ptr(), P->lev.ptr(), P->ent.ptr(), V, P->ee.ptr(), E));
        EULER_TRY(tour_successor_graph(ctx, P->ee.ptr(), E, sv));
        EULER_TRY(tour_components(ctx, sv, E, D));
        EULER_TRY(tour_circuit_vertices(ctx, D, E, C, cmap, nullptr, cnt));
        u64 ncirc = 0;
        EULER_TRY(read_u64(ctx, cnt, &ncirc));
        if (ncirc > 1) {
            euler_circuit_edge *cg = nullptr;
            u64 ncg = 0;
            EULER_TRY(tour_circuit_edges(ctx, P->ev.ptr(), P->ee.ptr(), P->ent.ptr(), V, D, cmap, E, &cg, &ncg));
            if (ncg) {
                DevTmp<u32> tree(ctx, ncg);
                TMP_CHECK(ctx, tree);
                u32 nt = 0;
                EULER_TRY(tour_spanning_forest(ctx, cg, ncg, (u32)ncirc, tree, &nt));
                EULER_TRY(tour_mark_spanning(ctx, cg, tree, nt, E, mark));
                EULER_TRY(tour_swipe(ctx, P->ev.ptr(), P->ent.ptr(), V, P->ee.ptr(), mark, E));
            }
        }
        char *d_text = nullptr;
        u64 bytes = 0, nc = 0;
        EULER_TRY(tour_emit_contigs(ctx, P->ev.ptr(), V, P->ee.ptr(), E, P->l, &d_text, &bytes, &nc,
                                    P->wide ? P->vkeys_hi.ptr() : nullptr));
        P->text_bytes = bytes; P->text_n = nc; P->text_valid = true; P->text_gen = ctx->text_gen;
        if (!out) {
            *out_bytes = bytes; *ncontigs = nc;
            return EULER_OK;
        }
    }
    const u64 bytes = P->text_bytes, nc = P->text_n;
    if (*out_bytes < bytes) return euler_fail(ctx, EULER_ERR_ARG, "contig buffer too small");
    if (bytes) {
        CUDA_TRY(ctx, cudaMemcpyAsync(out, ctx->text_buf.p, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    }
    *out_bytes = bytes; *ncontigs = nc;
    return EULER_OK;
}

// ---- FASTA / FASTQ ingestion on device (SURVEY §8 f1) ----------------------------------------------
int euler_ingest(euler_ctx *ctx, const char *file_bytes, uint64_t nbytes, int format, uint64_t *nreads, uint64_t *nbases)
{
    if (!ctx || !nreads || !nbases) return EULER_ERR_ARG;
    if (nbytes && !file_bytes) return euler_fail(ctx, EULER_ERR_ARG, "null file buffer");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    P->ingested = false;
    if (format == 0) {  // '>' opens a FASTA record, '@' a FASTQ record (eulercuda.py:469-476 goes by extension)
        format = 1;
        for (u64 i = 0; i < nbytes; i++) {
            const char c = file_bytes[i];
            if (c == '\n' || c == '\r' || c == ' ' || c == '\t') continue;
            format = (c == '@') ? 2 : 1;
            break;
        }
    }
    if (format != 1 && format != 2) return euler_fail(ctx, EULER_ERR_ARG, "format must be 0 (auto), 1 (FASTA) or 2 (FASTQ)");
    u64 nlines_ub = 1;
    for (u64 i = 0; i < nbytes; i++) nlines_ub += file_bytes[i] == '\n';
    DevTmp<unsigned char> d_file(ctx, nbytes + 16);
    TMP_CHECK(ctx, d_file);
    if (nbytes) CUDA_TRY(ctx, cudaMemcpyAsync(d_file.get(), file_bytes, nbytes, cudaMemcpyHostToDevice, ctx->stream));
    EULER_TRY(P->in_buf.reserve(ctx, nbytes + 16));
    EULER_TRY(P->in_off.reserve(ctx, nlines_ub + 2));
    u64 nr = 0, nb = 0;
    EULER_TRY(ingest_parse(ctx, d_file, nbytes, format == 2, P->in_buf.ptr(), P->in_off.ptr(), nlines_ub + 2, &nr, &nb));
    P->d_buf = P->in_buf.ptr(); P->d_off = P->in_off.ptr(); P->nreads = nr; P->n_bases = nb;
    P->ingested = true;
    *nreads = nr; *nbases = nb;
    return EULER_OK;
}

}  // extern "C"

int pipeline_resident_reads(euler_ctx *ctx, const void **d_buf, const u64 **d_off, u64 *nreads, u64 *n_bases)
{
    Pipeline *P = ctx->pipe;
    if (!P || !P->ingested) return euler_fail(ctx, EULER_ERR_STATE, "no reads resident: call euler_ingest first");
    *d_buf = P->in_buf.ptr(); *d_off = P->in_off.ptr(); *nreads = P->nreads; *n_bases = P->n_bases;
    return EULER_OK;
}

extern "C" {

int euler_ingest_download(euler_ctx *ctx, char *buf, uint64_t *read_off)
{
    if (!ctx) return EULER_ERR_ARG;
    const void *d_buf; const u64 *d_off; u64 nr, nb;
    EULER_TRY(pipeline_resident_reads(ctx, &d_buf, &d_off, &nr, &nb));
    if (buf && nb) CUDA_TRY(ctx, cudaMemcpyAsync(buf, d_buf, nb, cudaMemcpyDeviceToHost, ctx->stream));
    if (read_off) CUDA_TRY(ctx, cudaMemcpyAsync(read_off, d_off, (nr + 1) * sizeof(u64), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return EULER_OK;
}

int euler_pipeline_run_ingested(euler_ctx *ctx, uint32_t l, uint32_t flags, uint64_t distinct_hint, euler_stats *stats)
{
    if (!ctx) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    const void *d_buf; const u64 *d_off; u64 nr, nb;
    EULER_TRY(pipeline_resident_reads(ctx, &d_buf, &d_off, &nr, &nb));
    Pipeline *P = ctx->pipe;
    P->d_buf = d_buf; P->d_off = d_off; P->nreads = nr; P->n_bases = nb;
    return pipeline_run(ctx, P, l, flags, distinct_hint, stats);
}

// ---- multi-GPU: partition, (all-to-all by the caller), build ------------------------------------
int euler_dist_count(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases, uint32_t l,
                     uint32_t nranks, uint64_t *counts)
{
    if (!ctx || !counts) return EULER_ERR_ARG;
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,32]", l);
    if (nranks < 1 || nranks > 16) return euler_fail(ctx, EULER_ERR_ARG, "nranks %u out of range [1,16]", nranks);
    if (((uintptr_t)d_buf & 15) != 0) return euler_fail(ctx, EULER_ERR_ARG, "d_buf must be 16-byte aligned");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    EULER_TRY(P->stats.reserve(ctx, 64));
    EULER_TRY(P->start_bits.reserve(ctx, n_bases / 32 + 2));
    CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 64 * sizeof(u64), ctx->stream));
    EULER_TRY(enc_mark_starts(ctx, (const u64 *)d_read_off, nreads, n_bases, P->start_bits.ptr()));
    EULER_TRY(dist_partition(ctx, false, d_buf, n_bases, P->start_bits.ptr(), l, nranks, P->stats.ptr() + 32, nullptr, nullptr,
                             nullptr, 0));
    u64 h[18];
    EULER_TRY(read_u64s(ctx, P->stats.ptr() + 32, h, 18));
    for (u32 d = 0; d < nranks; d++) counts[d] = h[d];
    counts[nranks] = h[16];       // forward l-mer windows of this rank's reads
    counts[nranks + 1] = h[17];   // forward k-mer windows
    P->dist_bits_bases = n_bases; P->dist_bits_l = l;
    return EULER_OK;
}

int euler_dist_scatter(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                       uint32_t l, uint32_t nranks, void *d_send, const uint64_t *send_off)
{
    (void)d_read_off; (void)nreads;
    if (!ctx || !send_off || (!d_send && n_bases)) return EULER_ERR_ARG;
    if (nranks < 1 || nranks > 16) return euler_fail(ctx, EULER_ERR_ARG, "nranks %u out of range [1,16]", nranks);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,32]", l);
    if (((uintptr_t)d_buf & 15) != 0) return euler_fail(ctx, EULER_ERR_ARG, "d_buf must be 16-byte aligned");
    // the pass reuses the read-start bitmap of the count pass: it must be the one of these reads
    if (!P->start_bits.ptr() || P->dist_bits_bases != n_bases || P->dist_bits_l != l)
        return euler_fail(ctx, EULER_ERR_STATE, "euler_dist_scatter must follow euler_dist_count on the same reads and l");
    // cursors count from 0 inside each destination's segment, which starts at send_off[d]
    CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr() + 8, 0, 16 * sizeof(u64), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(P->stats.ptr() + 24, send_off, nranks * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    EULER_TRY(dist_partition(ctx, true, d_buf, n_bases, P->start_bits.ptr(), l, nranks, P->stats.ptr() + 32, P->stats.ptr() + 8,
                             (u64 *)d_send, P->stats.ptr() + 24, ~0ull));
    return EULER_OK;
}

// single pass: scatter into nranks fixed-capacity segments of d_send (segment d starts at d * seg_cap);
// counts[d] may exceed seg_cap, in which case the caller must redo the exchange with exact sizes
// shared tail of the two segment-scatter entry points.  seg_off: per destination, in KEYS from d_send
// (d_send == NULL: absolute address / key size).  Keys are 8 bytes for l <= 32, 16 bytes (wide_dist.cu) above.
static int scatter_to_segments(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                               uint32_t l, uint32_t nranks, void *d_send, const u64 *seg_off, uint64_t seg_cap, uint64_t *counts)
{
    if (l < 2 || l > 64) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,64]", l);
    if (nranks < 1 || nranks > (l > 32 ? 8u : 16u)) return euler_fail(ctx, EULER_ERR_ARG, "nranks %u out of range", nranks);
    if (((uintptr_t)d_buf & 15) != 0) return euler_fail(ctx, EULER_ERR_ARG, "d_buf must be 16-byte aligned");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    EULER_TRY(P->stats.reserve(ctx, 64));
    CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 64 * sizeof(u64), ctx->stream));
    CUDA_TRY(ctx, cudaMemcpyAsync(P->stats.ptr() + 24, seg_off, nranks * sizeof(u64), cudaMemcpyHostToDevice, ctx->stream));
    if (l > 32) {
        EULER_TRY(wide_dist_scatter(ctx, d_buf, (const u64 *)d_read_off, nreads, l, nranks, P->stats.ptr() + 32, P->stats.ptr() + 8,
                                    d_send, P->stats.ptr() + 24, seg_cap));
    } else {
        EULER_TRY(P->start_bits.reserve(ctx, n_bases / 32 + 2));
        P->dist_bits_bases = ~0ull;   // the bitmap no longer belongs to an euler_dist_count call
        EULER_TRY(enc_mark_starts(ctx, (const u64 *)d_read_off, nreads, n_bases, P->start_bits.ptr()));
        EULER_TRY(dist_partition(ctx, true, d_buf, n_bases, P->start_bits.ptr(), l, nranks, P->stats.ptr() + 32, P->stats.ptr() + 8,
                                 (u64 *)d_send, P->stats.ptr() + 24, seg_cap));
    }
    u64 h[16], w[2];
    EULER_TRY(read_u64s(ctx, P->stats.ptr() + 8, h, 16));
    EULER_TRY(read_u64s(ctx, P->stats.ptr() + 48, w, 2));
    for (u32 d = 0; d < nranks; d++) counts[d] = h[d];
    counts[nranks] = w[0];
    counts[nranks + 1] = w[1];
    return EULER_OK;
}

int euler_dist_scatter_segments(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                                uint32_t l, uint32_t nranks, void *d_send, uint64_t seg_cap, uint64_t *counts)
{
    if (!ctx || !counts || (!d_send && n_bases)) return EULER_ERR_ARG;
    u64 seg_off[16];
    for (u32 d = 0; d < 16; d++) seg_off[d] = (u64)d * seg_cap;
    return scatter_to_segments(ctx, d_buf, d_read_off, nreads, n_bases, l, nranks, d_send, seg_off, seg_cap, counts);
}

// ---- peer-memory exchange: the scatter kernel stores straight into the destination ranks' receive
// buffers over NVLink (CUDA IPC mappings), so the all-to-all is fused into the partition pass.
int euler_dist_recv_alloc(euler_ctx *ctx, uint64_t nkeys, void **dptr, unsigned char *handle64)
{
    if (!ctx || !dptr || !handle64) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    if (P->recv_buf && P->recv_cap < nkeys) {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(P->recv_buf);
        P->recv_buf = nullptr;
        P->recv_cap = 0;
    }
    if (!P->recv_buf) {
        // plain cudaMalloc: IPC handles cannot be taken from stream-ordered pool memory
        cudaError_t e = cudaMalloc(&P->recv_buf, (nkeys ? nkeys : 1) * sizeof(u64));
        if (e != cudaSuccess) return euler_fail(ctx, EULER_ERR_NOMEM, "cudaMalloc(recv %llu keys): %s", (u64)nkeys, cudaGetErrorString(e));
        P->recv_cap = nkeys;
    }
    cudaIpcMemHandle_t h;
    CUDA_TRY(ctx, cudaIpcGetMemHandle(&h, P->recv_buf));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &h, 64);
    *dptr = P->recv_buf;
    return EULER_OK;
}

int euler_dist_peer_open(euler_ctx *ctx, const unsigned char *handle64, void **dptr)
{
    if (!ctx || !dptr || !handle64) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    CUDA_TRY(ctx, cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess));
    return EULER_OK;
}

int euler_dist_peer_close(euler_ctx *ctx, void *dptr)
{
    if (!ctx) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaIpcCloseMemHandle(dptr));
    return EULER_OK;
}

// scatter with one destination pointer per rank (local or peer-mapped): region d receives at most
// seg_cap keys; counts as in euler_dist_scatter_segments
int euler_dist_scatter_peers(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                             uint32_t l, uint32_t nranks, void *const *dst_ptrs, uint64_t seg_cap, uint64_t *counts)
{
    if (!ctx || !counts || !dst_ptrs) return EULER_ERR_ARG;
    if (nranks < 1 || nranks > 16) return euler_fail(ctx, EULER_ERR_ARG, "nranks %u out of range [1,16]", nranks);
    const u64 key_bytes = l > 32 ? 16 : 8;
    u64 seg_off[16];
    for (u32 d = 0; d < nranks; d++) {
        if (((uintptr_t)dst_ptrs[d] & (key_bytes - 1)) != 0) return euler_fail(ctx, EULER_ERR_ARG, "destination pointer %u not key-aligned", d);
        seg_off[d] = (u64)(uintptr_t)dst_ptrs[d] / key_bytes;   // the kernel indexes keys from address 0
    }
    return scatter_to_segments(ctx, d_buf, d_read_off, nreads, n_bases, l, nranks, nullptr, seg_off, seg_cap, counts);
}

static int dist_build_impl(euler_ctx *ctx, const void *d_keys, uint64_t nkeys, uint32_t nregions, uint64_t region_stride,
                           const uint64_t *region_counts, uint32_t l, uint32_t rank, uint32_t nranks, uint64_t distinct_hint,
                           euler_stats *stats);

int euler_dist_build(euler_ctx *ctx, const void *d_keys, uint64_t nkeys, uint32_t l, uint32_t rank, uint32_t nranks,
                     uint64_t distinct_hint, euler_stats *stats)
{
    return dist_build_impl(ctx, d_keys, nkeys, 1, 0, &nkeys, l, rank, nranks, distinct_hint, stats);
}

// keys arrive in `nranks` regions of d_keys (region r starts at r * region_stride keys and holds region_counts[r] keys)
int euler_dist_build_regions(euler_ctx *ctx, const void *d_keys, uint64_t region_stride, const uint64_t *region_counts,
                             uint32_t l, uint32_t rank, uint32_t nranks, uint64_t distinct_hint, euler_stats *stats)
{
    if (!ctx || !region_counts) return EULER_ERR_ARG;
    u64 total = 0;
    for (u32 r = 0; r < nranks; r++) total += region_counts[r];
    return dist_build_impl(ctx, d_keys, total, nranks, region_stride, region_counts, l, rank, nranks, distinct_hint, stats);
}

static int dist_build_impl(euler_ctx *ctx, const void *d_keys, uint64_t nkeys, uint32_t nregions, uint64_t region_stride,
                           const uint64_t *region_counts, uint32_t l, uint32_t rank, uint32_t nranks, uint64_t distinct_hint,
                           euler_stats *stats)
{
    if (!ctx) return EULER_ERR_ARG;
    if (l < 2 || l > 64) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,64]", l);
    if (nranks < 1 || nranks > 16 || rank >= nranks) return euler_fail(ctx, EULER_ERR_ARG, "bad rank %u / %u", rank, nranks);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    if (l > 32) return wide_dist_build_impl(ctx, P, d_keys, nkeys, nregions, region_stride, region_counts, l, rank, nranks, distinct_hint, stats);
    cudaStream_t s = ctx->stream;
    const u32 k = l - 1;
    begin_run(P, l, 0, false, 0, 0);
    EULER_TRY(P->stats.reserve(ctx, 64));
    u64 lt_cap, vt_cap;
    caps_from_keys(P, nkeys, distinct_hint, lt_cap, vt_cap);
    u64 h[8] = {0};
    u32 retries = 0, launches = 0;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    while (true) {
        P->lt_cap = lt_cap; P->vt_cap = vt_cap;
        EULER_TRY(P->lt.reserve(ctx, lt_cap));
        EULER_TRY(P->lt_base.reserve(ctx, lt_cap)); EULER_TRY(P->lt_eoff.reserve(ctx, lt_cap));
        EULER_TRY(P->lt_own.reserve(ctx, lt_cap));
        EULER_TRY(P->vt_keys.reserve(ctx, vt_cap)); EULER_TRY(P->vt_id0.reserve(ctx, vt_cap));
        CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 8 * sizeof(u64), s));
        EULER_TRY(graph_table_clear(ctx, P->lt.keys(), P->lt.cnt(), lt_cap));
        EULER_TRY(graph_table_clear(ctx, P->vt_keys.ptr(), nullptr, vt_cap));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[4], s));
        // tables far larger than L2: regroup the keys by table region first (dist.cu, "L2 blocking")
        const u64 table_bytes = lt_cap * 12, block_min = (u64)dist_block_min_mb() << 20;
        const u32 cohash_l = use_cohash(block_min && table_bytes >= block_min) ? l : 0u;
        bool blocked = false;
        if (block_min && table_bytes >= block_min && nkeys >= 4096) {
            u32 nparts = (u32)((table_bytes + (48ull << 20) - 1) / (48ull << 20));
            if (nparts > 256) nparts = 256;
            const u64 part_cap = round_up(nkeys / nparts + nkeys / (nparts * 32ull) + 65536, 1024);
            u64 cur[256];
            if (P->blk_keys.reserve(ctx, (u64)nparts * part_cap) == EULER_OK && P->blk_cur.reserve(ctx, 256 + 8) == EULER_OK) {
                CUDA_TRY(ctx, cudaMemsetAsync(P->blk_cur.ptr(), 0, (256 + 8) * sizeof(u64), s));
                for (u32 r = 0; r < nregions; r++)
                    EULER_TRY(dist_block_keys(ctx, (const u64 *)d_keys + (u64)r * region_stride, region_counts[r], nparts,
                                              P->blk_cur.ptr(), P->blk_keys.ptr(), part_cap, cohash_l, P->blk_cur.ptr() + 256));
                u64 flag = 0;
                EULER_TRY(read_u64s(ctx, P->blk_cur.ptr(), cur, (int)nparts));
                EULER_TRY(read_u64(ctx, P->blk_cur.ptr() + 256, &flag));
                if (!flag) {
                    blocked = true;
                    for (u32 q = 0; q < nparts; q++)
                        EULER_TRY(dist_count_keys(ctx, P->blk_keys.ptr() + (u64)q * part_cap, cur[q], P->lt.keys(), P->lt.cnt(), lt_cap,
                                                  cohash_l, P->stats.ptr()));
                    launches += nregions + nparts;
                }
            } else {
                ctx->err.clear();   // no room for the regrouped copy: count in arrival order
            }
        }
        if (!blocked)
            for (u32 r = 0; r < nregions; r++)
                EULER_TRY(dist_count_keys(ctx, (const u64 *)d_keys + (u64)r * region_stride, region_counts[r], P->lt.keys(),
                                          P->lt.cnt(), lt_cap, cohash_l, P->stats.ptr()));
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
        EULER_TRY(dist_lt_scan(ctx, P->lt.keys(), P->lt.cnt(), lt_cap, l, rank, nranks, P->lt_base.ptr(),
                               P->lt_eoff.ptr(), P->lt_own.ptr(), P->stats.ptr() + 3));
        EULER_TRY(dist_vertex_insert(ctx, P->lt.keys(), lt_cap, l, P->vt_keys.ptr(), vt_cap, P->lt_own.ptr(),
                                     P->stats.ptr() + 2));
        EULER_TRY(graph_slot_scan(ctx, P->vt_keys.ptr(), vt_cap, k, P->vt_id0.ptr(), P->stats.ptr() + 4));
        launches += 4;
        EULER_TRY(read_u64s(ctx, P->stats.ptr(), h, 6));
        if ((h[2] & 3) == 0) break;
        if (++retries > 8) return euler_fail(ctx, EULER_ERR_OVERFLOW, "hash table overflow after %u regrows", retries);
        if (h[2] & 1) lt_cap *= 2;
        if (h[2] & 2) vt_cap *= 2;
    }
    const u64 U_l = h[3] & 0xffffffffull, V = h[4];
    u64 E = h[3] >> 32;
    // Every received key adds at most 2 to the edge total.  Past 2^32 the 32-bit offsets of the
    // reference layout (lmerOffsets, lstart / estart, EulerVertex.lp / .ep: `unsigned int`,
    // pydebruijn.py:90-101) cannot address the expanded edge arrays, which would not fit one GPU
    // either (32 B per edge): the compressed graph (keys, multiplicities, v1 / v2, degree slots) stays
    // exact, the offsets are kept modulo 2^32, and edge_count is the true 64-bit total.
    const char *force_big = getenv("EULER_B200_FORCE_BIG");   // test hook: take the 64-bit-total path on small inputs
    const bool big = 2 * nkeys >= 0xffffffffull || (force_big && atoi(force_big) == 1);
    P->U_l = U_l; P->V = V;
    if (V >= 0x3fffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "vertex count exceeds u32 ids");
    EULER_TRY(reserve_graph(ctx, P, U_l, V, false));
    EULER_TRY(clear_degrees(ctx, P, V, !big));   // paired degree regions: two sectors per l-mer instead of four
    EULER_TRY(graph_compact_vertices(ctx, P->vt_keys.ptr(), P->vt_id0.ptr(), vt_cap, k, P->vkeys.ptr()));
    VertexTable vt = {P->vt_keys.ptr(), P->vt_id0.ptr(), nullptr, vt_cap, k, TableHash{0, 0}};
    EULER_TRY(P->vt_bbase.reserve(ctx, vt_cap / EULER_BUCKET + 1));
    EULER_TRY(graph_bucket_bases(ctx, P->vt_id0.ptr(), vt_cap, P->vt_bbase.ptr()));
    vt.bbase = P->vt_bbase.ptr();
    EULER_TRY(dist_edges(ctx, P->lt.keys(), P->lt.cnt(), P->lt_base.ptr(), P->lt_eoff.ptr(), lt_cap, l, vt, P->lt_own.ptr(),
                         P->lkeys.ptr(), P->lvals.ptr(), P->loffs.ptr(), P->ev1.ptr(), P->ev2.ptr(), P->lcount.ptr(),
                         P->ecount.ptr(), big ? nullptr : P->deg.ptr()));
    if (!big) {
        EULER_TRY(graph_vertices_paired(ctx, P->deg.ptr(), k, P->vkeys.ptr(), V, P->lcount.ptr(), P->ecount.ptr(), P->lstart.ptr(),
                                        P->estart.ptr(), P->ev.ptr()));
        launches += 3;
    } else {
        // the pair scan would carry the overflow of one sum into the other: two u32 scans (wrapping), then D5
        EULER_TRY(scan_exclusive(ctx, ScanInU32{P->lcount.ptr()}, 4 * V, P->lstart.ptr(), (u64 *)nullptr));
        EULER_TRY(scan_exclusive(ctx, ScanInU32{P->ecount.ptr()}, 4 * V, P->estart.ptr(), (u64 *)nullptr));
        EULER_TRY(graph_setup_vertices(ctx, P->vkeys.ptr(), V, P->lcount.ptr(), P->lstart.ptr(), P->ecount.ptr(), P->estart.ptr(),
                                       P->ev.ptr()));
        EULER_TRY(graph_sum_u32(ctx, P->lvals.ptr(), U_l, P->stats.ptr() + 6));
        EULER_TRY(read_u64(ctx, P->stats.ptr() + 6, &E));
        launches += 6;
    }
    P->E = E;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[2], s));
    P->learned_bases = nkeys;
    // sizes for the next run of the same input: distinct canonical l-mers held by this rank (homed or
    // not; counted by the insert kernel) and canonical owned vertices (palindromes are rare)
    P->learned_lc = h[5] + h[5] / 32 + 16;
    P->learned_vc = (V + 1) / 2 + V / 32 + 16;
    P->st.n_lmer_windows = nkeys;
    return finish_run(ctx, P, lt_cap, vt_cap, retries, launches, 1, 2, stats);
}

// ---- multi-GPU form of the bucketed path -----------------------------------------------------------------------
// Every rank owns nb_per_rank buckets.  Pass 1 on every rank cuts its reads into records and stores them, as
// contiguous runs, into ONE stream per destination rank that lives in the destination's "area" (nranks streams of
// scap records, followed by the per-source record counts), published through a CUDA IPC handle; the local bucket id
// rides in the record header.  After a barrier the owner regroups its incoming streams into bucket regions (local
// memory) and runs pass 2 on them.  No key ever crosses the fabric: a 16-byte record carries ~7 l-mers.
static size_t bkt_stream_bytes(u32 nranks, u32 scap) { return (size_t)nranks * scap * 16; }

int euler_bkt_area_bytes(uint32_t nranks, uint32_t scap, uint64_t *bytes)
{
    if (!bytes) return EULER_ERR_ARG;
    *bytes = bkt_stream_bytes(nranks, scap) + (size_t)nranks * 8 + 256;
    return EULER_OK;
}

// which in {0, 1}: two areas per context so that a rank may scatter step i+1 while a peer still builds step i
int euler_bkt_area_alloc(euler_ctx *ctx, int which, uint32_t nranks, uint32_t scap, void **dptr, unsigned char *handle64)
{
    if (!ctx || !dptr || which < 0 || which > 1) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    uint64_t need = 0;
    euler_bkt_area_bytes(nranks, scap, &need);
    if (P->bk_area[which] && P->bk_area_bytes[which] < need) {
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(P->bk_area[which]);
        P->bk_area[which] = nullptr;
    }
    if (!P->bk_area[which]) {
        // plain cudaMalloc: IPC handles cannot be taken from stream-ordered pool memory
        cudaError_t e = cudaMalloc(&P->bk_area[which], need);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return euler_fail(ctx, EULER_ERR_NOMEM, "cudaMalloc(stream area %llu bytes): %s", (u64)need, cudaGetErrorString(e));
        }
        P->bk_area_bytes[which] = need;
    }
    if (handle64) {
        cudaIpcMemHandle_t h;
        CUDA_TRY(ctx, cudaIpcGetMemHandle(&h, P->bk_area[which]));
        memcpy(handle64, &h, 64);
    }
    *dptr = P->bk_area[which];
    return EULER_OK;
}

// out[0] N_l, out[1] N_k of this rank's reads, out[2] flags (BKT_FLAG_REGION = a stream overflowed), out[3] records in the fullest stream
int euler_bkt_scatter(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases, uint32_t l,
                      uint32_t my_rank, uint32_t nranks, uint32_t nb_per_rank, uint32_t scap, void *const *dst_areas, uint64_t *out,
                      void *d_out)
{
    if (!ctx || (!out && !d_out) || !dst_areas) return EULER_ERR_ARG;
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,32]", l);
    if (nranks < 1 || nranks > 16 || my_rank >= nranks || !nb_per_rank) return euler_fail(ctx, EULER_ERR_ARG, "bad rank / geometry");
    if (((uintptr_t)d_buf & 15) != 0) return euler_fail(ctx, EULER_ERR_ARG, "d_buf must be 16-byte aligned");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    cudaStream_t s = ctx->stream;
    EULER_TRY(P->stats.reserve(ctx, 64));
    EULER_TRY(P->start_bits.reserve(ctx, n_bases / 32 + 2));
    P->dist_bits_bases = ~0ull;   // the bitmap no longer belongs to an euler_dist_count call
    EULER_TRY(P->bk_scursors.reserve(ctx, 16));
    EULER_TRY(P->bk_dst.reserve(ctx, 16));
    uint4 *h_dst[16];
    for (u32 d = 0; d < nranks; d++) h_dst[d] = (uint4 *)dst_areas[d];
    CUDA_TRY(ctx, cudaMemcpyAsync(P->bk_dst.ptr(), h_dst, nranks * sizeof(uint4 *), cudaMemcpyHostToDevice, s));
    CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr() + 40, 0, 8 * sizeof(u64), s));
    CUDA_TRY(ctx, cudaMemsetAsync(P->bk_scursors.ptr(), 0, 16 * sizeof(u32), s));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[0], s));
    EULER_TRY(enc_mark_starts(ctx, (const u64 *)d_read_off, nreads, n_bases, P->start_bits.ptr()));
    EULER_TRY(bkt_partition_streams(ctx, d_buf, n_bases, P->start_bits.ptr(), l, nranks, nb_per_rank, my_rank, scap, P->bk_dst.ptr(),
                                    P->bk_scursors.ptr(), P->stats.ptr() + 40));
    EULER_TRY(bkt_push_counts(ctx, P->bk_scursors.ptr(), P->bk_dst.ptr(), bkt_stream_bytes(nranks, scap), nranks, my_rank, scap,
                              P->stats.ptr() + 46));
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[1], s));
    if (d_out) {   // asynchronous form: the four words stay on the device (e.g. as the payload of the caller's collective)
        CUDA_TRY(ctx, cudaMemcpyAsync(d_out, P->stats.ptr() + 40, 3 * sizeof(u64), cudaMemcpyDeviceToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync((u64 *)d_out + 3, P->stats.ptr() + 46, sizeof(u64), cudaMemcpyDeviceToDevice, s));
        P->bk_scatter_ms = -1.f;   // read from the events by the build call, after the stream has been synchronised
        return EULER_OK;
    }
    u64 h[8];
    EULER_TRY(read_u64s(ctx, P->stats.ptr() + 40, h, 8));
    out[0] = h[0]; out[1] = h[1]; out[2] = h[2]; out[3] = h[6];
    cudaEventElapsedTime(&P->bk_scatter_ms, ctx->ev[0], ctx->ev[1]);
    return EULER_OK;
}

// n_bases_hint: bases of the largest shard (sizes the bucket regions before anything has been learned; 0 = from scap)
int euler_bkt_build(euler_ctx *ctx, const void *d_area, uint32_t l, uint32_t my_rank, uint32_t nranks, uint32_t nb_per_rank,
                    uint32_t scap, uint64_t distinct_hint, euler_stats *stats)
{
    if (!ctx || !d_area) return EULER_ERR_ARG;
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [2,32]", l);
    if (nranks < 1 || nranks > 16 || my_rank >= nranks || !nb_per_rank) return euler_fail(ctx, EULER_ERR_ARG, "bad rank / geometry");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    Pipeline *P = get_pipe(ctx);
    cudaStream_t s = ctx->stream;
    begin_run(P, l, 0, false, 0, 0);
    EULER_TRY(P->stats.reserve(ctx, 64));
    const u32 nb = nb_per_rank;
    const u64 key = ((u64)nb << 32) ^ ((u64)nranks << 8) ^ l;   // what the learned capacities belong to
    const bool learned = P->bk_dist_key == key && P->bk_learned_u;
    const u64 est_c = distinct_hint ? distinct_hint : (learned ? (P->bk_learned_u + 1) / 2 : 0);
    u64 ucap = learned ? P->bk_learned_u + P->bk_learned_u / 32 + 1024 : (distinct_hint ? 2 * est_c + est_c / 4 + 1024 : 0);
    u64 vcap = learned ? P->bk_learned_v + P->bk_learned_v / 32 + 1024 : (distinct_hint ? 2 * est_c + est_c / 4 + 1024 : 0);
    u64 bcap = pow2_at_least((est_c ? est_c / 6 : (u64)nb * 64) + 1024);
    // bucket regions: what arrives is about one shard's worth of records, spread over nb buckets
    u32 rcap = learned && P->bk_dist_rcap ? P->bk_dist_rcap : (u32)((double)scap * nranks / 1.5 / nb * 1.5) + 64;
    u64 h[8] = {0};
    u32 retries = 0, launches = 0;
    u32 cap = (env_u32("EULER_B200_BKT_CAP", 1536) + 255u) / 256u * 256u;
    if (learned && P->bk_dist_cap > cap) cap = P->bk_dist_cap;
    if (P->bk_scatter_ms < 0.f) {   // asynchronous scatter: its events have completed by now (the caller synchronised on the exchange)
        if (cudaEventElapsedTime(&P->bk_scatter_ms, ctx->ev[0], ctx->ev[1]) != cudaSuccess) { P->bk_scatter_ms = 0.f; cudaGetLastError(); }
    }
    const u64 *d_counts = (const u64 *)((const char *)d_area + bkt_stream_bytes(nranks, scap));
    bool need_regroup = true;
    CUDA_TRY(ctx, cudaEventRecord(ctx->ev[7], s));
    while (true) {
        if ((u64)nb * rcap * 16 > (64ull << 30)) return euler_fail(ctx, EULER_ERR_NOMEM, "bucket regions of %u x %u records do not fit", nb, rcap);
        EULER_TRY(bkt_round(ctx, P, l, nb, rcap, cap, ucap, vcap, bcap, launches, h, [&]() -> int {
            CUDA_TRY(ctx, cudaMemsetAsync(P->stats.ptr(), 0, 8 * sizeof(u64), s));
            if (need_regroup) {
                CUDA_TRY(ctx, cudaMemsetAsync(P->bk_cursors.ptr(), 0, (size_t)nb * sizeof(u32), s));
                EULER_TRY(bkt_regroup(ctx, d_area, d_counts, nranks, scap, nb, rcap, P->bk_records.p, P->bk_cursors.ptr(), P->stats.ptr()));
                launches++;
                need_regroup = false;
            }
            return EULER_OK;
        }));
        const u64 fl = h[2];
        if ((fl & BKT_FLAG_TABLE) && cap * 2 > BKT_MAX_CAP)
            return euler_fail(ctx, EULER_ERR_OVERFLOW, "a bucket does not fit its shared-memory table: partition again with more buckets per rank");
        if (!(fl & (BKT_FLAG_REGION | BKT_FLAG_TABLE | BKT_FLAG_OUTPUT | BKT_FLAG_BOUNDARY))) break;
        if (++retries > 8) return euler_fail(ctx, EULER_ERR_OVERFLOW, "bucketed build: capacities did not settle");
        // every repair below is local to this rank (the streams stay where they are)
        if (fl & BKT_FLAG_REGION) { rcap = (u32)(h[6] + h[6] / 8 + 16); need_regroup = true; }   // stats[6] = the fullest bucket
        else if (fl & BKT_FLAG_TABLE) cap *= 2;   // larger tables, fewer resident blocks
        else if (fl & BKT_FLAG_OUTPUT) { ucap = h[3] + h[3] / 64 + 1024; vcap = h[4] + h[4] / 64 + 1024; }
        if (fl & BKT_FLAG_BOUNDARY) bcap *= 4;
    }
    const u64 U_l = h[3], V = h[4], E = h[5];
    if (V >= 0x3fffffffull || U_l >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "graph exceeds u32 ids (U_l=%llu V=%llu)", U_l, V);
    P->U_l = U_l; P->V = V; P->E = E;
    P->bk_dist_key = key; P->bk_learned_u = U_l; P->bk_learned_v = V; P->bk_dist_rcap = (u32)(h[6] + h[6] / 8 + 16);
    P->bk_dist_cap = cap;
    euler_stats &st = P->st;
    st.ms_count = P->bk_scatter_ms;   // the scatter pass of euler_bkt_scatter
    st.path = 1; st.n_buckets = nb; st.bucket_records = h[6]; st.redo_buckets = (u32)h[7];
    return finish_run(ctx, P, (u64)nb * cap, (u64)nb * cap, retries, launches, 7, 2, stats);
}

int euler_synth_reads_dev(euler_ctx *ctx, uint64_t genome_len, uint32_t read_len, uint32_t err_ppm, uint64_t first_read,
                          uint64_t nreads, void *d_out)
{
    if (!ctx || !d_out) return EULER_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return synth_reads(ctx, genome_len, read_len, err_ppm, first_read, nreads, d_out);
}

}  // extern "C"
