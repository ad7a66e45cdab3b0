// kernels.h -- internal device-pointer launchers (all asynchronous on ctx->stream).
#pragma once
#include "common.cuh"

// ---- encode.cu
int enc_mark_starts(euler_ctx *ctx, const u64 *d_off, u64 nreads, u64 n_bases, u32 *d_bits);
int enc_positions(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u64 *d_fwd, u64 *d_rc,
                  unsigned char *d_valid);
int enc_compute_kmers(euler_ctx *ctx, const u64 *d_lmers, u64 n, u64 mask, u64 *d_pk, u64 *d_sk);
// d_stats: [0] += forward l-windows, [1] += forward (l-1)-windows, [2] |= 1 on table overflow
int enc_count_canonical(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u64 *tab_keys,
                        u32 *tab_cnt, u64 cap, TableHash th, u64 *d_stats);

// merged count table (32-byte buckets {key, key, key, 3 x 21-bit counters}; cap_words = 4 * buckets)
int enc_merged_clear(euler_ctx *ctx, u64 *tab, u64 cap_words);
int enc_count_merged(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u64 *tab, u64 cap_words, bool cohash,
                     u64 *d_stats);
// -> SoA keys[cap_words] / cnt[cap_words] (slot 3 of every bucket empty)
int enc_merged_unpack(euler_ctx *ctx, const u64 *tab, u64 cap_words, u64 *keys, u32 *cnt);

// ---- graph.cu
// vertex-id lookup over the canonical k-mer table: id of strand 0 (canonical orientation) in id0,
// strand 1 in id1 (id1 == NULL: slot-order ids, strand 1 = id0 + 1)
struct VertexTable {
    const u64 *keys;
    const u32 *id0;
    const u32 *id1;
    u64 cap;
    u32 k;
    TableHash th;  // home rule of this table (plain or minimizer-ordered)
    const u32 *bbase = nullptr;  // slot-order ids only: id of the first strand of each bucket (common.cuh, table_find_id)
};
// plain key -> value table of the module-level API (pygpuhash TK/TV)
struct PlainTable {
    const u64 *keys;
    const u32 *vals;
    u64 cap;
};

int graph_table_clear(euler_ctx *ctx, u64 *keys, u32 *vals, u64 cap);
// insert canon(prefix) and canon(suffix) of every key of the canonical l-mer table
int graph_vertex_insert(euler_ctx *ctx, const u64 *lt_keys, u64 lt_cap, u32 l, u64 *vt_keys, u64 vt_cap, TableHash vth,
                        u64 *d_flags);
// exclusive scan of strand weights (0 empty / 1 palindrome / 2) over table slots
int graph_slot_scan(euler_ctx *ctx, const u64 *keys, u64 cap, u32 len, u32 *d_base, u64 *d_total);
// both-strand (key, multiplicity) pairs in slot order
int graph_compact_lmers(euler_ctx *ctx, const u64 *lt_keys, const u32 *lt_cnt, const u32 *lt_base, u64 lt_cap, u32 l,
                        u64 *lkeys, u32 *lvals);
// bbase[b] = id0[4 b]
int graph_bucket_bases(euler_ctx *ctx, const u32 *id0, u64 cap, u32 *bbase);
// both-strand vertex keys in slot order
int graph_compact_vertices(euler_ctx *ctx, const u64 *vt_keys, const u32 *vt_base, u64 vt_cap, u32 k, u64 *vkeys);
// id0/id1 of the table slot of each (sorted) vertex key: id = index in vkeys
int graph_assign_sorted_ids(euler_ctx *ctx, const u64 *vkeys, u64 nv, const u64 *vt_keys, u64 vt_cap, u32 k, TableHash vth,
                            u32 *id0, u32 *id1);
// D1 debruijnCount (+ compressed edges ev1/ev2) over explicit l-mer arrays
int graph_degree_slots(euler_ctx *ctx, const u64 *lkeys, const u32 *lvals, u64 nl, u32 l, const VertexTable &vt,
                       u32 *lcount, u32 *ecount, u32 *ev1, u32 *ev2);
int graph_degree_slots_plain(euler_ctx *ctx, const u64 *lkeys, const u32 *lvals, u64 nl, u32 l, const PlainTable &pt,
                             u64 nv, u32 *lcount, u32 *ecount);
// D5 setupVertices
int graph_setup_vertices(euler_ctx *ctx, const u64 *vkeys, u64 nv, const u32 *lcount, const u32 *lstart,
                         const u32 *ecount, const u32 *estart, euler_vertex *ev);
int graph_setup_vertices_plain(euler_ctx *ctx, const u64 *kmer_keys, u64 nk, const PlainTable &pt, u64 nv,
                               const u32 *lcount, const u32 *lstart, const u32 *ecount, const u32 *estart,
                               euler_vertex *ev);
// D6 setupEdges (expanded): ee / l[] / e[]
int graph_setup_edges(euler_ctx *ctx, const u64 *lkeys, const u32 *lvals, const u32 *loffs, u64 nl, u32 l,
                      const u32 *ev1, const u32 *ev2, const u32 *lstart, const u32 *estart, u32 ecount,
                      euler_edge *ee, u32 *lev, u32 *ent, const unsigned char *tf = nullptr);
int graph_setup_edges_plain(euler_ctx *ctx, const u64 *lkeys, const u32 *lvals, const u32 *loffs, u64 nl, u32 l,
                            const PlainTable &pt, const u32 *lstart, const u32 *estart, u32 ecount, euler_edge *ee,
                            u32 *lev, u32 *ent);
// *d_out = sum of v[0..n) as u64
int graph_sum_u32(euler_ctx *ctx, const u32 *v, u64 n, u64 *d_out);
// plain table build / lookup
int graph_plain_build(euler_ctx *ctx, const u64 *keys, const u32 *vals, u64 n, u64 *TK, u32 *TV, u64 cap, u64 *d_flags);
int graph_plain_lookup(euler_ctx *ctx, const PlainTable &pt, const u64 *q, u64 nq, u32 *out);
// (key,count) filter: keep count > limit, compact
int graph_filter_counts(euler_ctx *ctx, const u64 *keys, const u32 *vals, u64 n, u32 limit, u32 *d_base,
                        u64 *out_keys, u32 *out_vals, u64 *d_total);

// ---- tour.cu
int tour_reset_successors(euler_ctx *ctx, euler_edge *ee, u32 ecount);
int tour_assign_successor(euler_ctx *ctx, const euler_vertex *ev, const u32 *lev, const u32 *ent, u32 vcount,
                          euler_edge *ee, u32 ecount);
int tour_successor_graph(euler_ctx *ctx, const euler_edge *ee, u32 ecount, euler_succ_vertex *v);
int tour_components(euler_ctx *ctx, const euler_succ_vertex *v, u32 n, u32 *D);
int tour_circuit_vertices(euler_ctx *ctx, const u32 *D, u32 ecount, u32 *C, u32 *offset, u32 *cv, u64 *d_count);
// circuit edges, sorted; *out is a ctx-owned device array valid until the next call
int tour_circuit_edges(euler_ctx *ctx, const euler_vertex *ev, const euler_edge *ee, const u32 *ent, u32 vcount,
                       const u32 *D, const u32 *cmap, u32 ecount, euler_circuit_edge **out, u64 *count);
int tour_spanning_forest(euler_ctx *ctx, const euler_circuit_edge *cg, u64 cg_count, u32 cg_vcount, u32 *tree,
                         u32 *tree_count);
int tour_mark_spanning(euler_ctx *ctx, const euler_circuit_edge *cg, const u32 *tree, u32 tree_count, u32 ecount,
                       u32 *mark);
int tour_swipe(euler_ctx *ctx, const euler_vertex *ev, const u32 *ent, u32 vcount, euler_edge *ee, const u32 *mark,
               u32 ecount);
int tour_contig_starts(euler_ctx *ctx, const euler_edge *ee, u32 ecount, u32 *start);
// contig emission; *d_out ctx-owned device text, '\n'-terminated contigs
// vk_hi: high words of the vertex keys when k > 32 (wide.cu), else NULL
int tour_emit_contigs(euler_ctx *ctx, const euler_vertex *ev, u32 vcount, const euler_edge *ee, u32 ecount, u32 l,
                      char **d_out, u64 *out_bytes, u64 *ncontigs, const u64 *vk_hi = nullptr);

// ---- synth.cu
int synth_reads(euler_ctx *ctx, u64 G, u32 L, u32 err_ppm, u64 first, u64 nreads, void *d_out);

// ---- unitig.cu (K = 2..63; the key width follows from K there)
// unitigs of the reads (d_off[nreads + 1], B bases), text in ctx->text_buf.  cp == NULL: plain; else after the graph
// clean-up of clean.cu, with h_sums (host, sums_cap entries, may be NULL) the per-contig sums of the both-strand counts
// in output order
int unitigs_from_reads(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, u32 K, u32 limit,
                       const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                       euler_clean_stats *st);
// the same on a both-strand K-mer dictionary of n > 0 keys (low words d_lo, high words d_hi read for K > 32), all kept;
// with cp the counts must be both-strand counts
int unitigs_from_dict(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K,
                      const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                      euler_clean_stats *st);
// canonical count table (one-word keys, K <= 32) from a both-strand K-mer dictionary (keys, counts)
int unitig_dict_table(euler_ctx *ctx, const u64 *d_keys, const u32 *d_counts, u64 n, u32 K, u64 *tk, u32 *tc, u64 cap, u64 *d_flags);
// link graph of n contigs (text without separators, off[n+1]): links[16 i + 8 side + 2 base + (0 head '+' | 1 tail '-')]
int unitig_link_graph(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links);
// multi-k unitigs (the rule in euler_b200.h) of the reads for ks[0] < .. < ks[nk - 1]: the last step's text in
// ctx->text_buf, its sums in h_sums (may be NULL), one euler_multik_step per step in steps (may be NULL)
int unitigs_multik(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, const u32 *ks, u32 nk, u32 limit,
                   const euler_clean_params *params, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                   euler_multik_step *steps);

// clean_unitigs' output left on the device for the caller: contig i is ctx->text_buf[off[i], off[i + 1]) with its '\n'
// (off[ncontigs] = the text bytes), sums[i] its count sum; contigs from n_starts on are cycles.  The buffers grow only.
struct UnitigsKept {
    DevArr<u64> off, sums;
    u32 n_starts = 0;
};

// ---- clean.cu (key-independent): n nodes with forward extensions nbr[4 n], twin_id[n], both-strand counts cnt[n]
// (read only with rounds, sums or keep) and keys of key_stride 64-bit words each (low word first).  keep (may be NULL):
// leave offsets, sums and n_starts on the device as well
int clean_unitigs(euler_ctx *ctx, u32 n, u32 K, const u64 *key_words, u32 key_stride, const u32 *nbr, const u32 *twin_id,
                  const u32 *cnt, const euler_clean_params &p, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                  u64 sums_cap, euler_clean_stats *st, UnitigsKept *keep = nullptr);

// ---- graph.cu, fused fast path
// pair scan over l-mer table slots: base = distinct both-strand l-mer index, eoff = edge offset;
// *d_total_packed = (E << 32) | U_l
int graph_lt_scan(euler_ctx *ctx, const u64 *lt_keys, const u32 *lt_cnt, u64 cap, u32 l, u32 *base, u32 *eoff,
                  u64 *d_total_packed);
int graph_edges_fused(euler_ctx *ctx, const u64 *lt_keys, const u32 *lt_cnt, const u32 *base, const u32 *eoff, u64 cap,
                      u32 l, const VertexTable &vt, u64 *lkeys, u32 *lvals, u32 *loffs, u32 *ev1, u32 *ev2, u32 *lcount,
                      u32 *ecount, u32 *deg = nullptr);   // deg != NULL: paired degree regions (common.cuh) instead of lcount / ecount
int graph_vertices_fused(euler_ctx *ctx, const u32 *lcount, const u32 *ecount, const u64 *vkeys, u64 nv, u32 *lstart,
                         u32 *estart, euler_vertex *ev);
int graph_vertices_paired(euler_ctx *ctx, const u32 *deg, u32 k, const u64 *vkeys, u64 nv, u32 *lcount, u32 *ecount, u32 *lstart,
                          u32 *estart, euler_vertex *ev);

// ---- dist.cu (k-mer-space partition across GPUs)
// d_counts: 18 u64 ([0..15] keys per destination (count pass), [16] N_l, [17] N_k)
int dist_partition(euler_ctx *ctx, bool scatter, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u32 nranks,
                   u64 *d_counts, u64 *d_cursors, u64 *d_send, const u64 *d_seg_off, u64 seg_cap);
// cohash_l = l when the table is hashed by the canonical prefix k-mer (co-hashed tables), 0 = by the key
int dist_count_keys(euler_ctx *ctx, const u64 *d_keys, u64 n, u64 *tab_keys, u32 *tab_cnt, u64 cap, u32 cohash_l, u64 *d_stats);
// split keys into nparts runs of table-bucket ranges (out[part * part_cap + i]); d_cursors[nparts] = run lengths
int dist_block_keys(euler_ctx *ctx, const u64 *d_keys, u64 n, u32 nparts, u64 *d_cursors, u64 *d_out, u64 part_cap, u32 cohash_l,
                    u64 *d_flags);
int dist_vertex_insert(euler_ctx *ctx, const u64 *lt_keys, u64 lt_cap, u32 l, u64 *vt_keys, u64 vt_cap,
                       const unsigned char *own_flags, u64 *d_flags);
int dist_lt_scan(euler_ctx *ctx, const u64 *lt_keys, const u32 *lt_cnt, u64 cap, u32 l, u32 rank, u32 nranks, u32 *base,
                 u32 *eoff, unsigned char *own_flags, u64 *d_total_packed);
int dist_edges(euler_ctx *ctx, const u64 *lt_keys, const u32 *lt_cnt, const u32 *base, const u32 *eoff, u64 cap, u32 l,
               const VertexTable &vt, const unsigned char *own_flags, u64 *lkeys, u32 *lvals, u32 *loffs, u32 *ev1, u32 *ev2,
               u32 *lcount, u32 *ecount, u32 *deg = nullptr);

// ---- packed.cu (L2-sized quotient table for the count kernel)
int enc_count_packed(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u64 *tab, u32 b,
                     u64 *side_keys, u32 *side_cnt, u64 side_cap, u64 *d_stats);
int enc_unpack(euler_ctx *ctx, const u64 *tab, u32 b, const u64 *side_keys, const u32 *side_cnt, u64 side_cap, u64 *d_side_used,
               u64 *keys, u32 *cnt);

// ---- ingest.cu (FASTA / FASTQ parsing on device)
int ingest_parse(euler_ctx *ctx, const unsigned char *d_file, u64 n, int fastq, unsigned char *d_reads, u64 *d_off, u64 off_cap,
                 u64 *nreads, u64 *nbases);
// reads left resident by euler_ingest (pipeline.cu)
int pipeline_resident_reads(euler_ctx *ctx, const void **d_buf, const u64 **d_off, u64 *nreads, u64 *n_bases);

// ---- bucket_part.cu / bucket_build.cu (minimizer-bucketed hot path, bucket.cuh)
// flags of stats[2] raised by the bucketed kernels
#define BKT_FLAG_REGION 0x10ull     // a (bucket, source) record region overflowed: rerun with the capacity of stats[6]
#define BKT_FLAG_TABLE 0x20ull      // a bucket's shared-memory table filled up: rerun with more buckets
#define BKT_FLAG_OUTPUT 0x40ull     // the artefact arrays were too small: rerun with the totals of stats[3..5]
#define BKT_FLAG_BOUNDARY 0x80ull   // the cross-bucket edge table filled up
#define BKT_FLAG_INTERNAL 0x100ull  // a consistency check failed (pushed degree totals != looked-up degree slots)
// pass 1: records of this rank's reads into the regions (local bucket, source rank) of every owner;
// d_dst[r] = base of rank r's record area, d_cursors[nranks * nb_per_rank] (zeroed by the caller) counts per global bucket;
// d_stats: [0] += N_l, [1] += N_k, [2] |= flags
int bkt_partition(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u32 nranks, u32 nb_per_rank, u32 my_rank,
                  u32 rcap, uint4 *const *d_dst, u32 *d_cursors, u64 *d_stats);
// pass 2 over the nb local buckets
#define BKT_MAX_CAP 7424u   // 29 B per slot: the largest per-bucket table that fits one block's shared memory
#define BKT_REDO_CAP 128u   // buckets the second pass of the build can take over from the first
struct BktBuild {
    const void *records;   // region (b, src) at ((b * nranks + src) * rcap) records of 16 bytes
    const u32 *counts;     // [nb * nranks]
    u32 nb, nranks, rcap, l, cap;   // cap: slots of each per-bucket shared-memory table (l-mers, vertices), a multiple of 256
    u64 *lkeys; u32 *lvals, *loffs, *ev1, *ev2; u64 ucap;
    u64 *vkeys; u32 *lcount, *ecount, *lstart, *estart; euler_vertex *ev; u64 vcap;
    void *state;           // bkt_state_bytes(nb)
    u64 *bkeys; u32 *bvals; u64 bcap;   // cross-bucket edge table: bcap keys (power of two), 2 * bcap values
    u64 *stats;            // [2] |= flags, [3] U_l, [4] V, [5] E, [6] max records in a region, [7] buckets redone by the second pass
};
int bkt_build(euler_ctx *ctx, const BktBuild &B);
size_t bkt_state_bytes(u32 nb);
size_t bkt_build_smem(u32 cap);
// canonical-id post-processing of the bucketed build
int bkt_iota(euler_ctx *ctx, u32 *v, u64 n);
int bkt_invert_perm(euler_ctx *ctx, const u32 *perm, u64 n, u32 *inv);
int bkt_gather_rows(euler_ctx *ctx, const u32 *perm, u64 n, const u32 *a_in, const u32 *b_in, u32 *a_out, u32 *b_out);
int bkt_gather_edges(euler_ctx *ctx, const u32 *perm, u64 n, const u32 *newid, const u32 *lvals, const u32 *ev1, const u32 *ev2,
                     u32 *lvals_out, u32 *ev1_out, u32 *ev2_out);
// multi-GPU stream form of pass 1 (one stream per destination rank, the local bucket id in bits 8..31 of the record header),
// the count hand-over and the owner-side regrouping of the incoming streams into bucket regions
int bkt_partition_streams(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, u32 nranks, u32 nb_per_rank,
                          u32 my_rank, u32 scap, uint4 *const *d_dst, u32 *d_cursors, u64 *d_stats);
int bkt_push_counts(euler_ctx *ctx, const u32 *d_cursors, uint4 *const *d_dst, u64 stream_bytes, u32 nranks, u32 my_rank, u32 scap, u64 *d_max);
int bkt_regroup(euler_ctx *ctx, const void *d_streams, const u64 *d_counts, u32 nranks, u32 scap, u32 nb, u32 rcap, void *d_records,
                u32 *d_cursors, u64 *d_stats);
