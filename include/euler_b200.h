/*
 * euler_b200.h -- C ABI of libeuler_b200.so: the B200-native (sm_100a) drop-in for the
 * data-parallel assembly front end of zenlc2000/pycuda-euler (encode -> hash -> de Bruijn graph
 * -> Euler tour / components -> partial contigs).
 *
 * The reference has no FFI of its own: its boundary is the Python function surface of the five
 * PyCUDA "operator" modules plus eulercuda.py (SURVEY.md §8b).  Every entry point below names the
 * reference wrapper (file:line under src/eulercuda/) it replaces; the ctypes binding a maintainer
 * would add is shown in INTEGRATION.md and implemented in pycuda-euler_b200/_native.py.
 *
 * Conventions
 *   - plain pointers and sizes only; all functions return EULER_OK (0) or a negative error code;
 *     euler_last_error(ctx) gives the message.  The caller owns every host buffer; the library
 *     owns device memory behind the opaque euler_ctx.  One ctx per (thread, GPU); a ctx is not
 *     thread-safe.  All work is issued on the ctx stream.
 *   - "host" entry points take host pointers and copy in/out inside the call (what the reference
 *     wrappers do, e.g. pyencode.py:85-92).  "dev" entry points take device pointers and are
 *     asynchronous on the ctx stream unless they return a count.
 *   - 2-bit code: A=0 C=1 G=2 T=3 (case-insensitive), MSB-first (pyencode.py:42,64-71).  Any other
 *     byte ends the current window run (referenceAssembler.py:29); windows never cross a read
 *     boundary (SURVEY B1).  k-mer = vertex = (l-1)-mer, l-mer = edge (eulercuda.py:554 -> :450).
 *   - ids are u32 (vertices < 2^30, distinct l-mers < 2^32).  E (= sum of multiplicities) is reported as 64 bits; past
 *     2^32 the compressed graph stays exact, the reference's `unsigned int` offsets are kept modulo 2^32 and the expanded
 *     edge arrays (EULER_RUN_EXPAND_EDGES) are refused -- the reference's own limit (SURVEY 2.3).
 */
#ifndef EULER_B200_H
#define EULER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EULER_OK 0
#define EULER_ERR_CUDA (-1)      /* CUDA runtime error */
#define EULER_ERR_ARG (-2)       /* bad argument (NULL, l out of range, ...) */
#define EULER_ERR_NOMEM (-3)     /* device or host allocation failed */
#define EULER_ERR_RANGE (-4)     /* result does not fit u32 ids (E >= 2^32) */
#define EULER_ERR_STATE (-5)     /* call made in the wrong pipeline state */
#define EULER_ERR_OVERFLOW (-6)  /* hash table overflow that could not be repaired */
#define EULER_ERR_NOGPU (-7)     /* no CUDA device: there is no CPU fallback */

typedef struct euler_ctx euler_ctx;

/* device-ABI structs, identical to the reference numpy dtypes */
typedef struct { uint64_t vid; uint32_t ep, ecount, lp, lcount; } euler_vertex;   /* pydebruijn.py:197-203,:607 */
typedef struct { uint64_t eid; uint32_t v1, v2, s, pad; } euler_edge;             /* pydebruijn.py:345-351,:605 */
typedef struct { uint32_t vid, n1, n2; } euler_succ_vertex;                       /* pyeulertour.py:127-131,:735 */
typedef struct { uint32_t ceid, e1, e2, c1, c2; } euler_circuit_edge;             /* pyeulertour.py:421-427,:786 */

/* ---- context (replaces `import pycuda.autoinit`, pyencode.py:3) ---------------------------- */
int euler_ctx_create(int device, euler_ctx **out);
void euler_ctx_destroy(euler_ctx *ctx);
const char *euler_last_error(const euler_ctx *ctx);
/* use an existing CUDA stream (cudaStream_t as void*), e.g. torch.cuda.current_stream().cuda_stream */
int euler_ctx_set_stream(euler_ctx *ctx, void *cuda_stream);
int euler_ctx_sync(euler_ctx *ctx);
int euler_version(void);

/* =========================================================================================
 * Stage-wise entry points on HOST buffers (module-level parity with the L3 wrappers)
 * ======================================================================================= */

/* pyencode.encode_lmer_device (:16) + compute_lmer_complement_device (:164).
 * buf: B = read_off[nreads] bytes; out_fwd/out_rc/out_valid: B entries, indexed by window START
 * byte; entries without a valid window are 0.  out_rc / out_valid may be NULL.  l in [1,32]. */
int euler_encode_lmers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads,
                       uint32_t l, uint64_t *out_fwd, uint64_t *out_rc, uint8_t *out_valid);

/* pyencode.compute_kmer_device (:103): pk = (lmer & (mask<<2))>>2, sk = lmer & mask */
int euler_compute_kmers(euler_ctx *ctx, const uint64_t *lmers, uint64_t n, uint64_t kmer_mask,
                        uint64_t *pkmers, uint64_t *skmers);

/* eulercuda.readLmersKmersCuda (:74-180): distinct l-mers + multiplicities and distinct k-mers over
 * both strands, ascending key order, k-mer value = rank.  Two-call protocol: call with all output
 * pointers NULL to get the counts, then with buffers of at least that size. */
int euler_count_lmers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads,
                      uint32_t l, uint64_t *lmer_count, uint64_t *kmer_count,
                      uint64_t *lmer_keys, uint32_t *lmer_values, uint64_t *kmer_keys, uint32_t *kmer_values);

/* Both-strand multiset of len-mers (== referenceAssembler.build(reads, len, limit) :25-42, as
 * (key,count) pairs with count > limit), ascending.  Same two-call protocol. len in [1,32]. */
int euler_count_mers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads,
                     uint32_t len, uint32_t limit, uint64_t *count, uint64_t *keys, uint32_t *values);
/* euler_count_mers on two-word keys: bits 0..63 of each key in keys_lo, bits 64..127 in keys_hi, ascending in
 * (hi, lo) order.  len in [1,64]; for len <= 32 keys_hi is all zero and the rest equals euler_count_mers.  Keys
 * are canonical in the table, so len = 64 is counted although its poly-T key is all ones.  Same two-call protocol. */
int euler_count_mers_wide(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads,
                          uint32_t len, uint32_t limit, uint64_t *count, uint64_t *keys_lo, uint64_t *keys_hi,
                          uint32_t *values);

/* pygpuhash.create_hash_table_device (:262) / phase1 (:19) / copy_to_bucket (:77) / bucket_sort (:174):
 * open-addressing table.  capacity = euler_hash_capacity(n); TK/TV have `capacity` entries, empty
 * slots hold key 0xFFFFFFFFFFFFFFFF / value 0xFFFFFFFF. */
uint64_t euler_hash_capacity(uint64_t n);
int euler_hash_build(euler_ctx *ctx, const uint64_t *keys, const uint32_t *values, uint64_t n,
                     uint64_t capacity, uint64_t *TK, uint32_t *TV);
/* pydebruijn getHashValue (:57-88): out[i] = value or 0xffffffff */
int euler_hash_lookup(euler_ctx *ctx, const uint64_t *TK, const uint32_t *TV, uint64_t capacity,
                      const uint64_t *queries, uint64_t nq, uint32_t *out);

/* pycuda.scan.ExclusiveScanKernel(uintc,"a+b",0) call sites (pygpuhash.py:290, pydebruijn.py:560-573,
 * pyeulertour.py:748,774) */
int euler_exclusive_scan_u32(euler_ctx *ctx, const uint32_t *in, uint64_t n, uint32_t *out);

/* pydebruijn.debruijn_count_device (:16): lcount/ecount have 4*vertex_count entries (zeroed here) */
int euler_debruijn_count(euler_ctx *ctx, const uint64_t *lmer_keys, const uint32_t *lmer_values,
                         uint64_t lmer_count, const uint64_t *TK, const uint32_t *TV, uint64_t capacity,
                         uint32_t l, uint64_t vertex_count, uint32_t *lcount, uint32_t *ecount);
/* pydebruijn.setup_vertices_device (:182) */
int euler_setup_vertices(euler_ctx *ctx, const uint64_t *kmer_keys, uint64_t kmer_count,
                         const uint64_t *TK, const uint32_t *TV, uint64_t capacity,
                         const uint32_t *lcount, const uint32_t *lstart, const uint32_t *ecount,
                         const uint32_t *estart, euler_vertex *ev);
/* pydebruijn.setup_edges_device (:327): ee/l/e have edge_count = sum(lmer_values) entries */
int euler_setup_edges(euler_ctx *ctx, const uint64_t *lmer_keys, const uint32_t *lmer_values,
                      const uint32_t *lmer_offsets, uint64_t lmer_count, const uint64_t *TK,
                      const uint32_t *TV, uint64_t capacity, uint32_t l, const uint32_t *lstart,
                      const uint32_t *estart, uint64_t edge_count, euler_edge *ee, uint32_t *lev, uint32_t *ent);

/* pyeulertour.assign_successor_device (:18): ee updated in place */
int euler_assign_successor(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *lev, const uint32_t *ent,
                           uint32_t vcount, euler_edge *ee, uint32_t ecount);
/* pyeulertour.construct_successor_graphP1/P2_device (:110,:165) */
int euler_successor_graph(euler_ctx *ctx, const euler_edge *ee, uint32_t ecount, euler_succ_vertex *v);
/* pycomponent.find_component_device (:676), run to its fix-point: D[i] = min node id of i's component */
int euler_find_components(euler_ctx *ctx, const euler_succ_vertex *v, uint32_t n, uint32_t *D);
/* pyeulertour.calculate_circuit_graph_vertex_data_device (:220) + scan (:748) + construct_circuit_Graph_vertex
 * (:269): C[ecount], offset[ecount] (exclusive scan of C), cv[*count] */
int euler_circuit_vertices(euler_ctx *ctx, const uint32_t *D, uint32_t ecount, uint32_t *C,
                           uint32_t *offset, uint32_t *cv, uint32_t *count);
/* pyeulertour.calculate_circuit_graph_edge_data (:308) + assign_circuit_graph_edge_data (:394) + the host
 * sort (:792).  Two-call protocol on `out` (NULL -> count only). Sorted by (c1,c2,ceid,e1,e2). */
int euler_circuit_edges(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *ent, uint32_t vcount,
                        const uint32_t *D, const uint32_t *cmap, uint32_t ecount,
                        euler_circuit_edge *out, uint64_t *count);
/* eulercuda.findSpanningTree (:267): indices of the spanning-forest circuit edges (Kruskal in index order) */
int euler_spanning_forest(euler_ctx *ctx, const euler_circuit_edge *cg, uint64_t cg_count, uint32_t cg_vcount,
                          uint32_t *tree, uint32_t *tree_count);
/* pyeulertour.mark_spanning_euler_edges (:587): mark[ecount], zeroed here */
int euler_mark_spanning(euler_ctx *ctx, const euler_circuit_edge *cg, uint64_t cg_count, const uint32_t *tree,
                        uint32_t tree_count, uint32_t ecount, uint32_t *mark);
/* pyeulertour.execute_swipe (:496): ee updated in place */
int euler_swipe(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *ent, uint32_t vcount, euler_edge *ee,
                const uint32_t *mark, uint32_t ecount);
/* pyeulertour.identify_contig_start (:668) */
int euler_contig_starts(euler_ctx *ctx, const euler_edge *ee, uint32_t ecount, uint32_t *start);
/* eulercuda.generatePartialContig (:329) host walk, on device (list ranking + scatter).
 * out: '\n'-terminated contigs in the reference's order; two-call protocol (out NULL -> sizes). */
int euler_emit_contigs(euler_ctx *ctx, const euler_vertex *ev, uint32_t vcount, const euler_edge *ee,
                       uint32_t ecount, uint32_t l, char *out, uint64_t *out_bytes, uint64_t *ncontigs);

/* referenceAssembler.build (:25-42) + all_contigs (:79-88) on device: unitigs of the both-strand
 * K-mer graph restricted to K-mers with count > limit.  Each unitig is written once, in one of its
 * two orientations; isolated cycles start at an implementation-chosen node.  '\n'-terminated
 * contigs; two-call protocol on out (NULL -> sizes).  K in [2,63]: K > 32 runs on two-word keys.
 * K = 64 is refused because the two-word tables mark an empty slot with all ones, which is the
 * poly-T 64-mer; every K-mer of K <= 63 bases leaves the top two bits of its high word clear. */
int euler_unitigs(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t K,
                  uint32_t limit, char *out, uint64_t *out_bytes, uint64_t *ncontigs);

/* referenceAssembler.all_contigs(d, k) (:79-88) on a K-mer dictionary, i.e. on the output of build /
 * euler_count_mers: keys[n] (either strand or both; they are canonicalised), counts[n] (both-strand counts, every
 * key present).  Output as euler_unitigs. */
int euler_unitigs_from_kmers(euler_ctx *ctx, const uint64_t *keys, const uint32_t *counts, uint64_t n, uint32_t K,
                             char *out, uint64_t *out_bytes, uint64_t *ncontigs);
/* the same on two-word keys (keys_lo / keys_hi as euler_count_mers_wide returns them).  K in [2,63]; for
 * K <= 32 only keys_lo is read (keys_hi may be NULL) and the result is that of euler_unitigs_from_kmers. */
int euler_unitigs_from_kmers_wide(euler_ctx *ctx, const uint64_t *keys_lo, const uint64_t *keys_hi, const uint32_t *counts,
                                  uint64_t n, uint32_t K, char *out, uint64_t *out_bytes, uint64_t *ncontigs);
/* Link graph G of referenceAssembler.all_contigs (:90-111) for n contigs: text = the contigs back to back
 * (no separators), off[n+1].  links: u32[16 n]; entry [16 i + 8 side + 2 base + o]: side 0 = candidates
 * fw(last K-mer of contig i), side 1 = fw(twin(first K-mer)); base = A,C,G,T; o = 0: contig whose head is the
 * candidate ('+'), o = 1: contig whose twin(tail) is ('-'); 0xffffffff = none.  When two contigs share a head
 * (or a twin(tail)), the later one is reported, as in the reference's dicts.  K in [2,63]: K >= 32 uses
 * two-word end tables (the one-word tables' EMPTY key is the poly-T 32-mer; see euler_unitigs for 63). */
int euler_unitig_links(euler_ctx *ctx, const char *text, const uint64_t *off, uint64_t n, uint32_t K, uint32_t *links);

/* =========================================================================================
 * Fused device-resident pipeline (the measured hot path)
 * ======================================================================================= */
typedef struct {
    uint64_t n_reads, n_bases;
    uint64_t n_kmer_windows;      /* forward k-mer windows  N_k (the metric's unit) */
    uint64_t n_lmer_windows;      /* forward l-mer windows  N_l */
    uint64_t distinct_lmers;      /* U_l, both strands */
    uint64_t distinct_kmers;      /* U_k = vertex count, both strands */
    uint64_t edge_count;          /* E = 2 N_l */
    uint64_t lmer_table_capacity, kmer_table_capacity;
    uint32_t retries;             /* table regrow-and-rerun count */
    float ms_count, ms_graph, ms_total;   /* CUDA-event times of the last run: table init + count | graph | both */
    float ms_count_kernel;                /* the fused encode+count kernel alone */
    uint32_t kernel_launches;             /* kernels of this library launched by the run */
    /* bucketed path (path == 1): the partition pass is ms_count_kernel, the per-bucket build ms_build_kernel */
    float ms_build_kernel;
    uint32_t path;                        /* 0 = global-table path (round 1), 1 = minimizer-bucketed path */
    uint32_t n_buckets;                   /* buckets of the last run */
    uint32_t redo_buckets;     /* bucketed path: buckets rebuilt by the second pass (they overflowed the first pass's tables) */
    uint64_t bucket_records;              /* largest number of 16-byte records in one bucket region */
} euler_stats;

#define EULER_RUN_EXPAND_EDGES 1u   /* also materialise ee[] / l[] / e[] (needs E < 2^32) */
#define EULER_RUN_CANONICAL_IDS 2u  /* ids = rank in ascending key order (sort), else slot order */

/* reads already resident in device memory (d_buf: n_bases ASCII bytes, 16-byte aligned;
 * d_read_off: nreads+1 u64).  distinct_hint = expected distinct canonical l-mers (0 = estimate).
 * l in [2,64].  The reference stops at 64-bit keys (KEY_T, pyencode.py:22-33: l <= 32); for
 * l in 33..64 (k up to 63, BASELINE.json configs[4]) keys are two words: the low words are the
 * usual artefacts, the high words EULER_ART_*_KEYS_HI, and contigs come out the same way. */
int euler_pipeline_run_dev(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads,
                           uint64_t n_bases, uint32_t l, uint32_t flags, uint64_t distinct_hint,
                           euler_stats *stats);
/* same, from host buffers (H2D copy inside the call) */
int euler_pipeline_run_host(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads,
                            uint32_t l, uint32_t flags, uint64_t distinct_hint, euler_stats *stats);

/* the graph stage on an existing l-mer table instead of reads -- e.g. the per-rank tables of the partitioned
 * path joined on one GPU (assembler.py): keys[n] (either strand or both; canonicalised), counts[n] = both-strand
 * multiplicities.  l in [2,32].  Artefacts and contigs as after euler_pipeline_run_host. */
int euler_pipeline_run_lmers(euler_ctx *ctx, const uint64_t *keys, const uint32_t *counts, uint64_t n, uint32_t l,
                             uint32_t flags, euler_stats *stats);

/* artefacts of the last run */
enum {
    EULER_ART_LMER_KEYS = 0,   /* u64[U_l] */
    EULER_ART_LMER_VALUES = 1, /* u32[U_l] */
    EULER_ART_LMER_OFFSETS = 2,/* u32[U_l] exclusive scan of values */
    EULER_ART_KMER_KEYS = 3,   /* u64[U_k], id = index */
    EULER_ART_LCOUNT = 4,      /* u32[4 U_k] */
    EULER_ART_ECOUNT = 5,
    EULER_ART_LSTART = 6,
    EULER_ART_ESTART = 7,
    EULER_ART_EV = 8,          /* euler_vertex[U_k] */
    EULER_ART_EDGE_V1 = 9,     /* u32[U_l] compressed edges: prefix vertex */
    EULER_ART_EDGE_V2 = 10,    /* u32[U_l] suffix vertex */
    EULER_ART_EE = 11,         /* euler_edge[E]  (EXPAND_EDGES) */
    EULER_ART_LEV = 12,        /* u32[E] l[]      (EXPAND_EDGES) */
    EULER_ART_ENT = 13,        /* u32[E] e[]      (EXPAND_EDGES) */
    EULER_ART_LMER_KEYS_HI = 14, /* u64[U_l] bits 64..127 of the l-mer keys; only after a run with l > 32 */
    EULER_ART_KMER_KEYS_HI = 15  /* u64[U_k] bits 64..127 of the vertex keys; euler_vertex.vid holds the low word */
};
int euler_pipeline_artifact_bytes(euler_ctx *ctx, int which, uint64_t *bytes);
int euler_pipeline_download(euler_ctx *ctx, int which, void *host_dst, uint64_t cap_bytes);
/* device pointer of an artefact (valid until the next run) */
int euler_pipeline_device_ptr(euler_ctx *ctx, int which, void **dptr);

/* Euler tour + contigs on the resident graph (needs EXPAND_EDGES); two-call protocol on out */
int euler_pipeline_contigs(euler_ctx *ctx, char *out, uint64_t *out_bytes, uint64_t *ncontigs);

/* =========================================================================================
 * FASTA / FASTQ ingestion on device (replaces eulercuda.read_fasta :439-447 / read_fastq :44-56):
 * the raw file bytes are parsed on the GPU (line split, header / '+' / quality skipping, read
 * offsets) and the reads stay resident for the calls below.  format: 0 auto, 1 FASTA, 2 FASTQ.
 * FASTA: every line not starting with '>' is one read; FASTQ: lines with index % 4 == 1.
 * ======================================================================================= */
int euler_ingest(euler_ctx *ctx, const char *file_bytes, uint64_t nbytes, int format, uint64_t *nreads,
                 uint64_t *nbases);
/* copy the parsed reads back: buf nbases bytes, read_off nreads + 1 entries (either may be NULL) */
int euler_ingest_download(euler_ctx *ctx, char *buf, uint64_t *read_off);
int euler_pipeline_run_ingested(euler_ctx *ctx, uint32_t l, uint32_t flags, uint64_t distinct_hint,
                                euler_stats *stats);
int euler_unitigs_ingested(euler_ctx *ctx, uint32_t K, uint32_t limit, char *out, uint64_t *out_bytes,
                           uint64_t *ncontigs);

/* =========================================================================================
 * k-mer-space partition across the GPUs of one box (one process per GPU; the caller owns the
 * collective, e.g. torch.distributed all_to_all_single over NCCL).  The reference has no analogue:
 * its only parallelism is Spark mapPartitions over read partitions (src/cli_spark_gpu.py:37).
 *   1. euler_dist_count    per-destination key counts of this rank's reads
 *   2. euler_dist_scatter  write the canonical l-mer keys, grouped by destination rank
 *   3. (all-to-all of the u64 keys)
 *   4. euler_dist_build    count the received keys and build this rank's part of the graph; the
 *                          artefacts are read with euler_pipeline_download (local ids; v2 of an edge
 *                          whose suffix vertex lives on another rank is 0xffffffff)
 * ======================================================================================= */
/* counts: nranks + 2 entries: keys for rank 0..nranks-1, then this rank's forward l-mer and k-mer windows */
int euler_dist_count(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads,
                     uint64_t n_bases, uint32_t l, uint32_t nranks, uint64_t *counts);
/* d_send: u64[sum counts]; send_off[r] = first index of rank r's keys (exclusive scan of counts) */
int euler_dist_scatter(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads,
                       uint64_t n_bases, uint32_t l, uint32_t nranks, void *d_send, const uint64_t *send_off);
/* single-pass form of count + scatter: segment d of d_send starts at d * seg_cap keys; counts has
 * nranks + 2 entries as above; counts[d] > seg_cap means that segment overflowed (redo with exact sizes) */
int euler_dist_scatter_segments(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads,
                                uint64_t n_bases, uint32_t l, uint32_t nranks, void *d_send, uint64_t seg_cap,
                                uint64_t *counts);
/* Peer-memory exchange (fuses the all-to-all into the scatter pass): every rank allocates a receive
 * buffer of nranks * seg_cap keys, publishes its CUDA IPC handle (64 bytes), opens the others', and
 * scatters with dst_ptrs[d] = (rank d's buffer) + my_rank * seg_cap.  After a barrier and an
 * exchange of the counts, euler_dist_build_regions counts the nranks regions of the local buffer. */
int euler_dist_recv_alloc(euler_ctx *ctx, uint64_t nkeys, void **dptr, unsigned char *handle64);
int euler_dist_peer_open(euler_ctx *ctx, const unsigned char *handle64, void **dptr);
int euler_dist_peer_close(euler_ctx *ctx, void *dptr);
int euler_dist_scatter_peers(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads,
                             uint64_t n_bases, uint32_t l, uint32_t nranks, void *const *dst_ptrs,
                             uint64_t seg_cap, uint64_t *counts);
int euler_dist_build_regions(euler_ctx *ctx, const void *d_keys, uint64_t region_stride,
                             const uint64_t *region_counts, uint32_t l, uint32_t rank, uint32_t nranks,
                             uint64_t distinct_hint, euler_stats *stats);
int euler_dist_build(euler_ctx *ctx, const void *d_keys, uint64_t nkeys, uint32_t l, uint32_t rank,
                     uint32_t nranks, uint64_t distinct_hint, euler_stats *stats);

/* =========================================================================================
 * Multi-GPU form of the minimizer-bucketed hot path (csrc/bucket.cuh).  Replaces, for l <= 32, the key
 * exchange above: what crosses NVLink is the 2-bit packed minimizer runs of the reads (16-byte records of up
 * to 17 l-mers), not one 8-byte key per l-mer.  The reference has no analogue (src/cli_spark_gpu.py:37 assembles
 * every read partition on its own).
 *   geometry (the same on every rank): nranks, nb_per_rank buckets owned by each rank, scap records per
 *   (destination, source) stream.  Vertex v belongs to bucket(minimizer(v)); rank = bucket / nb_per_rank, the
 *   round-1 owner rule.
 *   1. euler_bkt_area_alloc   a receive area (two per context, `which` = step parity) + its CUDA IPC handle:
 *                             nranks streams of scap records, then the per-source record counts
 *   2. euler_bkt_scatter      one pass over this rank's reads: per tile one contiguous run of records per destination,
 *                             stored straight into the owners' streams (dst_areas[r] = rank r's area, local or
 *                             peer-mapped); the local bucket id rides in the record header
 *   3. (barrier across ranks)
 *   4. euler_bkt_build        regroup the incoming streams into bucket regions (local), then the per-bucket
 *                             shared-memory build; artefacts as after euler_dist_build (local ids; v2 = 0xffffffff
 *                             when the suffix vertex lives on another rank).  Every repair (region, table or
 *                             output capacity) is local to the rank.
 * ======================================================================================= */
int euler_bkt_area_bytes(uint32_t nranks, uint32_t scap, uint64_t *bytes);
int euler_bkt_area_alloc(euler_ctx *ctx, int which, uint32_t nranks, uint32_t scap, void **dptr, unsigned char *handle64);
/* out[0] forward l-mer windows, out[1] forward k-mer windows of this rank's reads, out[2] flags (0x10: a stream
 * overflowed -- scatter again with the capacity of out[3]), out[3] records in the fullest stream.
 * d_out != NULL: asynchronous form, the four words are left in device memory (u64[4]) on the ctx stream and `out`
 * may be NULL -- e.g. as the payload of the collective that doubles as the barrier of step 3 */
int euler_bkt_scatter(euler_ctx *ctx, const void *d_buf, const void *d_read_off, uint64_t nreads, uint64_t n_bases,
                      uint32_t l, uint32_t my_rank, uint32_t nranks, uint32_t nb_per_rank, uint32_t scap,
                      void *const *dst_areas, uint64_t *out, void *d_out);
int euler_bkt_build(euler_ctx *ctx, const void *d_area, uint32_t l, uint32_t my_rank, uint32_t nranks,
                    uint32_t nb_per_rank, uint32_t scap, uint64_t distinct_hint, euler_stats *stats);

/* =========================================================================================
 * Step-level entry points of the reference's fine-grained wrappers (kept for callers; the
 * product path uses the open-addressing table and union-find components instead)
 * ======================================================================================= */
/* pygpuhash.phase1_device (:19): offset[i] = arrival order of key i in bucket hash_h(key), count[] += */
int euler_compat_phase1(euler_ctx *ctx, const uint64_t *keys, uint64_t n, uint32_t bucketCount,
                        uint32_t *offset, uint32_t *count);
/* pygpuhash.copy_to_bucket_device (:77) */
int euler_compat_copy_to_bucket(euler_ctx *ctx, const uint64_t *keys, const uint32_t *values,
                                const uint32_t *offset, uint64_t n, const uint32_t *start,
                                uint32_t bucketCount, uint64_t *bufferK, uint32_t *bufferV);
/* pygpuhash.bucket_sort_device (:174): TK/TV have bucketCount*520 entries */
int euler_compat_bucket_sort(euler_ctx *ctx, const uint64_t *bufferK, const uint32_t *bufferV, uint64_t n,
                             const uint32_t *start, const uint32_t *bucketSize, uint32_t bucketCount,
                             uint64_t *TK, uint32_t *TV);
/* pycomponent sub-steps (:17-:654). step: 0 init, 1 s1p1, 2 s1p2, 3 s2p1, 4 s2p2, 5 s3p1, 6 s3p2,
 * 7 s4p1, 8 s4p2, 9 s5.  Arrays are in/out, n entries each (NULL = zeroed scratch); flag: one u32 */
int euler_compat_cc_step(euler_ctx *ctx, int step, uint32_t n, uint32_t s, const euler_succ_vertex *v,
                         uint32_t *prevD, uint32_t *D, uint32_t *Q, uint32_t *t1, uint32_t *val1,
                         uint32_t *t2, uint32_t *val2, uint32_t *flag);

/* =========================================================================================
 * Deterministic synthetic reads on device (SURVEY §8d), L bytes per read, no separators
 * ======================================================================================= */
int euler_synth_reads_dev(euler_ctx *ctx, uint64_t genome_len, uint32_t read_len, uint32_t err_ppm,
                          uint64_t first_read, uint64_t nreads, void *d_out);

#ifdef __cplusplus
}
#endif
#endif /* EULER_B200_H */
