// api.cu -- stage-wise C-ABI entry points on HOST buffers.  Each one uploads its inputs, runs the
// device kernels and downloads its outputs inside the call, which is exactly the contract of the
// reference's L3 wrappers (one H2D/D2H round trip per wrapper, e.g. pyencode.py:85-92).
#include "kernels.h"
#include "scan.cuh"
#include "sort.cuh"
#include "tmp.cuh"
#include "wide.cuh"

template <typename T>
static int upload(euler_ctx *ctx, DevTmp<T> &d, const T *h, u64 n)
{
    if (!d.ok()) return euler_fail(ctx, EULER_ERR_NOMEM, "device temp alloc failed: %s", cudaGetErrorString(d.err));
    if (n) {
        if (!h) return euler_fail(ctx, EULER_ERR_ARG, "null host input");
        CUDA_TRY(ctx, cudaMemcpyAsync(d.get(), h, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    }
    return EULER_OK;
}
template <typename T>
static int download(euler_ctx *ctx, T *h, const T *d, u64 n)
{
    if (n && h) CUDA_TRY(ctx, cudaMemcpyAsync(h, d, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
    return EULER_OK;
}
#define ENTER(ctx)                                                  \
    if (!(ctx)) return EULER_ERR_ARG;                               \
    CUDA_TRY((ctx), cudaSetDevice((ctx)->device))
#define FINISH(ctx)                                                 \
    CUDA_TRY((ctx), cudaStreamSynchronize((ctx)->stream));          \
    return EULER_OK

extern "C" {

uint64_t euler_hash_capacity(uint64_t n)
{
    u64 c = (u64)((double)(n < 16 ? 16 : n) / 0.55) + 1;
    return (c + 1023) / 1024 * 1024;
}

int euler_encode_lmers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t l,
                       uint64_t *out_fwd, uint64_t *out_rc, uint8_t *out_valid)
{
    ENTER(ctx);
    if (!read_off || !out_fwd) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (l < 1 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l-mer length %u out of range [1,32]", l);
    const u64 B = read_off[nreads];
    if (!B) return EULER_OK;
    DevTmp<unsigned char> d_buf(ctx, B + 16);
    DevTmp<u64> d_off(ctx, nreads + 1), d_fwd(ctx, B), d_rc(ctx, out_rc ? B : 1);
    DevTmp<u32> d_bits(ctx, B / 32 + 2);
    DevTmp<unsigned char> d_valid(ctx, out_valid ? B : 1);
    TMP_CHECK(ctx, d_fwd); TMP_CHECK(ctx, d_rc); TMP_CHECK(ctx, d_bits); TMP_CHECK(ctx, d_valid);
    EULER_TRY(upload(ctx, d_buf, (const unsigned char *)buf, B));
    EULER_TRY(upload(ctx, d_off, (const u64 *)read_off, nreads + 1));
    EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    EULER_TRY(enc_positions(ctx, d_buf, B, d_bits, l, d_fwd, out_rc ? d_rc.get() : nullptr, out_valid ? d_valid.get() : nullptr));
    EULER_TRY(download(ctx, (u64 *)out_fwd, d_fwd.get(), B));
    if (out_rc) EULER_TRY(download(ctx, (u64 *)out_rc, d_rc.get(), B));
    if (out_valid) EULER_TRY(download(ctx, out_valid, d_valid.get(), B));
    FINISH(ctx);
}

int euler_compute_kmers(euler_ctx *ctx, const uint64_t *lmers, uint64_t n, uint64_t kmer_mask, uint64_t *pkmers,
                        uint64_t *skmers)
{
    ENTER(ctx);
    if (!n) return EULER_OK;
    if (!pkmers || !skmers) return euler_fail(ctx, EULER_ERR_ARG, "null output");
    DevTmp<u64> d_l(ctx, n), d_p(ctx, n), d_s(ctx, n);
    TMP_CHECK(ctx, d_p); TMP_CHECK(ctx, d_s);
    EULER_TRY(upload(ctx, d_l, (const u64 *)lmers, n));
    EULER_TRY(enc_compute_kmers(ctx, d_l, n, kmer_mask, d_p, d_s));
    EULER_TRY(download(ctx, (u64 *)pkmers, d_p.get(), n));
    EULER_TRY(download(ctx, (u64 *)skmers, d_s.get(), n));
    FINISH(ctx);
}

int euler_count_lmers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t l,
                      uint64_t *lmer_count, uint64_t *kmer_count, uint64_t *lmer_keys, uint32_t *lmer_values,
                      uint64_t *kmer_keys, uint32_t *kmer_values)
{
    ENTER(ctx);
    if (!lmer_count || !kmer_count) return euler_fail(ctx, EULER_ERR_ARG, "null count pointers");
    const u64 cap_l = *lmer_count, cap_k = *kmer_count;
    euler_stats st;
    EULER_TRY(euler_pipeline_run_host(ctx, buf, read_off, nreads, l, EULER_RUN_CANONICAL_IDS, 0, &st));
    *lmer_count = st.distinct_lmers;
    *kmer_count = st.distinct_kmers;
    if (lmer_keys || lmer_values || kmer_keys || kmer_values) {
        if (cap_l < st.distinct_lmers || cap_k < st.distinct_kmers)
            return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small (%llu/%llu < %llu/%llu)", cap_l, cap_k,
                              (u64)st.distinct_lmers, (u64)st.distinct_kmers);
        if (lmer_keys) EULER_TRY(euler_pipeline_download(ctx, EULER_ART_LMER_KEYS, lmer_keys, cap_l * 8));
        if (lmer_values) EULER_TRY(euler_pipeline_download(ctx, EULER_ART_LMER_VALUES, lmer_values, cap_l * 4));
        if (kmer_keys) EULER_TRY(euler_pipeline_download(ctx, EULER_ART_KMER_KEYS, kmer_keys, cap_k * 8));
        if (kmer_values) for (u64 i = 0; i < st.distinct_kmers; i++) kmer_values[i] = (u32)i;  // value = rank
    }
    return EULER_OK;
}

int euler_count_mers(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t len,
                     uint32_t limit, uint64_t *count, uint64_t *keys, uint32_t *values)
{
    ENTER(ctx);
    if (!read_off || !count) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (len < 1 || len > 32) return euler_fail(ctx, EULER_ERR_ARG, "mer length %u out of range [1,32]", len);
    const u64 out_cap = *count;
    *count = 0;
    const u64 B = read_off[nreads];
    if (!B) return EULER_OK;
    DevTmp<unsigned char> d_buf(ctx, B + 16);
    DevTmp<u64> d_off(ctx, nreads + 1), d_stats(ctx, 8);
    DevTmp<u32> d_bits(ctx, B / 32 + 2);
    TMP_CHECK(ctx, d_bits); TMP_CHECK(ctx, d_stats);
    EULER_TRY(upload(ctx, d_buf, (const unsigned char *)buf, B));
    EULER_TRY(upload(ctx, d_off, (const u64 *)read_off, nreads + 1));
    EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    u64 cap = euler_hash_capacity(B);
    DevTmp<u64> tk(ctx, cap);
    DevTmp<u32> tc(ctx, cap), base(ctx, cap);
    TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc); TMP_CHECK(ctx, base);
    CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, 8 * sizeof(u64), ctx->stream));
    EULER_TRY(graph_table_clear(ctx, tk, tc, cap));
    EULER_TRY(enc_count_canonical(ctx, d_buf, B, d_bits, len, tk, tc, cap, TableHash{0, 0}, d_stats));
    EULER_TRY(graph_slot_scan(ctx, tk, cap, len, base, d_stats.get() + 3));
    u64 h[4];
    EULER_TRY(read_u64s(ctx, d_stats, h, 4));
    if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
    const u64 U = h[3];
    if (!U) return EULER_OK;
    DevTmp<u64> lk(ctx, U), lk2(ctx, U);
    DevTmp<u32> lv(ctx, U), lv2(ctx, U), fbase(ctx, U);
    const u32 nblocks = (u32)((U + RS_TILE - 1) / RS_TILE);
    DevTmp<u32> hist(ctx, (u64)256 * nblocks);
    TMP_CHECK(ctx, lk); TMP_CHECK(ctx, lk2); TMP_CHECK(ctx, lv); TMP_CHECK(ctx, lv2); TMP_CHECK(ctx, fbase); TMP_CHECK(ctx, hist);
    EULER_TRY(graph_compact_lmers(ctx, tk, tc, base, cap, len, lk, lv));
    EULER_TRY(radix_sort_pairs(ctx, lk, lv, U, 2 * (int)len, lk2, lv2, hist));
    EULER_TRY(graph_filter_counts(ctx, lk, lv, U, limit, fbase, lk2, lv2, d_stats.get() + 4));
    u64 kept = 0;
    EULER_TRY(read_u64(ctx, d_stats.get() + 4, &kept));
    *count = kept;
    if (keys || values) {
        if (out_cap < kept) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small (%llu < %llu)", out_cap, kept);
        EULER_TRY(download(ctx, (u64 *)keys, lk2.get(), kept));
        EULER_TRY(download(ctx, values, lv2.get(), kept));
    }
    FINISH(ctx);
}

// euler_count_mers on two-word keys: len in [1,64]; len <= 32 is euler_count_mers with keys_hi all zero
int euler_count_mers_wide(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t len,
                          uint32_t limit, uint64_t *count, uint64_t *keys_lo, uint64_t *keys_hi, uint32_t *values)
{
    ENTER(ctx);
    if (!read_off || !count) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (len < 1 || len > 64) return euler_fail(ctx, EULER_ERR_ARG, "mer length %u out of range [1,64]", len);
    const u64 out_cap = *count;
    if (len <= 32) {
        EULER_TRY(euler_count_mers(ctx, buf, read_off, nreads, len, limit, count, keys_lo, values));
        if (keys_hi) {
            if (out_cap < *count) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small (%llu < %llu)", out_cap, *count);
            for (u64 i = 0; i < *count; i++) keys_hi[i] = 0;
        }
        return EULER_OK;
    }
    *count = 0;
    const u64 B = read_off[nreads];
    if (!B) return EULER_OK;
    DevTmp<unsigned char> d_buf(ctx, B + 16);
    DevTmp<u64> d_off(ctx, nreads + 1), d_stats(ctx, 8);
    DevTmp<u32> d_bits(ctx, B / 32 + 2);
    TMP_CHECK(ctx, d_bits); TMP_CHECK(ctx, d_stats);
    EULER_TRY(upload(ctx, d_buf, (const unsigned char *)buf, B));
    EULER_TRY(upload(ctx, d_off, (const u64 *)read_off, nreads + 1));
    EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    const u64 cap = euler_hash_capacity(B);
    DevTmp<K128> tk(ctx, cap);
    DevTmp<u32> tc(ctx, cap), base(ctx, cap);
    TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc); TMP_CHECK(ctx, base);
    CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, 8 * sizeof(u64), ctx->stream));
    EULER_TRY(wide_table_clear(ctx, tk, tc, cap));
    EULER_TRY(wide_count_tiled(ctx, d_buf, B, d_bits, len, tk, tc, cap, d_stats));
    EULER_TRY(wide_slot_scan(ctx, tk, cap, len, base, d_stats.get() + 3));
    u64 h[4];
    EULER_TRY(read_u64s(ctx, d_stats, h, 4));
    if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
    const u64 U = h[3];
    if (!U) return EULER_OK;
    DevTmp<u64> lo(ctx, U), hi(ctx, U), lo2(ctx, U), hi2(ctx, U);
    DevTmp<u32> lv(ctx, U), lv2(ctx, U), fbase(ctx, U);
    TMP_CHECK(ctx, lo); TMP_CHECK(ctx, hi); TMP_CHECK(ctx, lo2); TMP_CHECK(ctx, hi2); TMP_CHECK(ctx, lv); TMP_CHECK(ctx, lv2);
    TMP_CHECK(ctx, fbase);
    EULER_TRY(wide_compact_lmers(ctx, tk, tc, base, cap, len, lo, hi, lv));
    EULER_TRY(wide_sort(ctx, lo, hi, lv, U, 2 * (int)len));
    EULER_TRY(wide_filter_counts(ctx, lo, hi, lv, U, limit, fbase, lo2, hi2, lv2, d_stats.get() + 4));
    u64 kept = 0;
    EULER_TRY(read_u64(ctx, d_stats.get() + 4, &kept));
    *count = kept;
    if (keys_lo || keys_hi || values) {
        if (out_cap < kept) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small (%llu < %llu)", out_cap, kept);
        EULER_TRY(download(ctx, (u64 *)keys_lo, lo2.get(), kept));
        EULER_TRY(download(ctx, (u64 *)keys_hi, hi2.get(), kept));
        EULER_TRY(download(ctx, values, lv2.get(), kept));
    }
    FINISH(ctx);
}

static int unitigs_core(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, uint32_t K, uint32_t limit,
                        char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    const u64 cap_out = *out_bytes;
    *out_bytes = 0; *ncontigs = 0;
    if (!B) return EULER_OK;
    DevTmp<u64> d_stats(ctx, 8);
    DevTmp<u32> d_bits(ctx, B / 32 + 2);
    TMP_CHECK(ctx, d_bits); TMP_CHECK(ctx, d_stats);
    EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    const u64 cap = euler_hash_capacity(B);
    CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, 8 * sizeof(u64), ctx->stream));
    char *d_text = nullptr;
    u64 bytes = 0, nc = 0, nn = 0;
    if (K > 32) {
        // two-word keys: the tiled 128-bit count of the pipeline (wide.cu) into a K128 table of the same capacity
        DevTmp<K128> tk(ctx, cap);
        DevTmp<u32> tc(ctx, cap);
        TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc);
        EULER_TRY(wide_table_clear(ctx, tk, tc, cap));
        EULER_TRY(wide_count_tiled(ctx, d_buf, B, d_bits, K, tk, tc, cap, d_stats));
        u64 h[3];
        EULER_TRY(read_u64s(ctx, d_stats, h, 3));
        if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
        EULER_TRY(wide_unitig_from_table(ctx, tk, tc, cap, K, limit, &d_text, &bytes, &nc, &nn));
    } else {
        DevTmp<u64> tk(ctx, cap);
        DevTmp<u32> tc(ctx, cap);
        TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc);
        EULER_TRY(graph_table_clear(ctx, tk, tc, cap));
        EULER_TRY(enc_count_canonical(ctx, d_buf, B, d_bits, K, tk, tc, cap, TableHash{0, 0}, d_stats));
        u64 h[3];
        EULER_TRY(read_u64s(ctx, d_stats, h, 3));
        if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
        EULER_TRY(unitig_from_table(ctx, tk, tc, cap, K, limit, &d_text, &bytes, &nc, &nn));
    }
    *out_bytes = bytes; *ncontigs = nc;
    if (out) {
        if (cap_out < bytes) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small");
        EULER_TRY(download(ctx, out, (const char *)d_text, bytes));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return EULER_OK;
}

int euler_unitigs(euler_ctx *ctx, const char *buf, const uint64_t *read_off, uint64_t nreads, uint32_t K, uint32_t limit,
                  char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    ENTER(ctx);
    if (!read_off || !out_bytes || !ncontigs) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (K < 2 || K > 63) return euler_fail(ctx, EULER_ERR_ARG, "K %u out of range [2,63]", K);
    const u64 B = read_off[nreads];
    DevTmp<unsigned char> d_buf(ctx, B + 16);
    DevTmp<u64> d_off(ctx, nreads + 1);
    EULER_TRY(upload(ctx, d_buf, (const unsigned char *)buf, B));
    EULER_TRY(upload(ctx, d_off, (const u64 *)read_off, nreads + 1));
    return unitigs_core(ctx, d_buf, d_off, nreads, B, K, limit, out, out_bytes, ncontigs);
}

// unitigs of the reads left on the device by euler_ingest
int euler_unitigs_ingested(euler_ctx *ctx, uint32_t K, uint32_t limit, char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    ENTER(ctx);
    if (!out_bytes || !ncontigs) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (K < 2 || K > 63) return euler_fail(ctx, EULER_ERR_ARG, "K %u out of range [2,63]", K);
    const void *d_buf; const u64 *d_off; u64 nr, nb;
    EULER_TRY(pipeline_resident_reads(ctx, &d_buf, &d_off, &nr, &nb));
    return unitigs_core(ctx, d_buf, d_off, nr, nb, K, limit, out, out_bytes, ncontigs);
}

// referenceAssembler.all_contigs(d, k) :79-88 on a K-mer dictionary (the output of build / euler_count_mers)
int euler_unitigs_from_kmers(euler_ctx *ctx, const uint64_t *keys, const uint32_t *counts, uint64_t n, uint32_t K, char *out,
                             uint64_t *out_bytes, uint64_t *ncontigs)
{
    ENTER(ctx);
    if (!out_bytes || !ncontigs || (n && (!keys || !counts))) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (K < 2 || K > 32) return euler_fail(ctx, EULER_ERR_ARG, "K %u out of range [2,32]", K);
    const u64 cap_out = *out_bytes;
    *out_bytes = 0; *ncontigs = 0;
    if (!n) return EULER_OK;
    const u64 cap = euler_hash_capacity(n);
    DevTmp<u64> dk(ctx, n), tk(ctx, cap), flags(ctx, 1);
    DevTmp<u32> dc(ctx, n), tc(ctx, cap);
    TMP_CHECK(ctx, dk); TMP_CHECK(ctx, dc); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc); TMP_CHECK(ctx, flags);
    EULER_TRY(upload(ctx, dk, (const u64 *)keys, n));
    EULER_TRY(upload(ctx, dc, counts, n));
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(graph_table_clear(ctx, tk, tc, cap));
    EULER_TRY(unitig_dict_table(ctx, dk, dc, n, K, tk, tc, cap, flags));
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "K-mer table full");
    char *d_text = nullptr;
    u64 bytes = 0, nc = 0, nn = 0;
    EULER_TRY(unitig_from_table(ctx, tk, tc, cap, K, 0, &d_text, &bytes, &nc, &nn));
    *out_bytes = bytes; *ncontigs = nc;
    if (out) {
        if (cap_out < bytes) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small");
        EULER_TRY(download(ctx, out, (const char *)d_text, bytes));
    }
    FINISH(ctx);
}

// euler_unitigs_from_kmers on two-word keys: K in [2,63]; K <= 32 reads keys_lo only (keys_hi may be NULL)
int euler_unitigs_from_kmers_wide(euler_ctx *ctx, const uint64_t *keys_lo, const uint64_t *keys_hi, const uint32_t *counts,
                                  uint64_t n, uint32_t K, char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    ENTER(ctx);
    if (K < 2 || K > 63) return euler_fail(ctx, EULER_ERR_ARG, "K %u out of range [2,63]", K);
    if (K <= 32) return euler_unitigs_from_kmers(ctx, keys_lo, counts, n, K, out, out_bytes, ncontigs);
    if (!out_bytes || !ncontigs || (n && (!keys_lo || !keys_hi || !counts))) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    const u64 cap_out = *out_bytes;
    *out_bytes = 0; *ncontigs = 0;
    if (!n) return EULER_OK;
    const u64 cap = euler_hash_capacity(n);
    DevTmp<u64> dlo(ctx, n), dhi(ctx, n), flags(ctx, 1);
    DevTmp<u32> dc(ctx, n), tc(ctx, cap);
    DevTmp<K128> tk(ctx, cap);
    TMP_CHECK(ctx, dlo); TMP_CHECK(ctx, dhi); TMP_CHECK(ctx, dc); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc); TMP_CHECK(ctx, flags);
    EULER_TRY(upload(ctx, dlo, (const u64 *)keys_lo, n));
    EULER_TRY(upload(ctx, dhi, (const u64 *)keys_hi, n));
    EULER_TRY(upload(ctx, dc, counts, n));
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(wide_table_clear(ctx, tk, tc, cap));
    EULER_TRY(wide_unitig_dict_table(ctx, dlo, dhi, dc, n, K, tk, tc, cap, flags));
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "K-mer table full");
    char *d_text = nullptr;
    u64 bytes = 0, nc = 0, nn = 0;
    EULER_TRY(wide_unitig_from_table(ctx, tk, tc, cap, K, 0, &d_text, &bytes, &nc, &nn));
    *out_bytes = bytes; *ncontigs = nc;
    if (out) {
        if (cap_out < bytes) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small");
        EULER_TRY(download(ctx, out, (const char *)d_text, bytes));
    }
    FINISH(ctx);
}

// link graph G of referenceAssembler.all_contigs :90-111 for n contigs (text: the contigs back to back, no
// separators; off[n+1]).  links: u32[16 n], entry [16 i + 8 side + 2 base + o]: side 0 = successors of the last
// K-mer, side 1 = of twin(first K-mer); o = 0: the hit is a contig head ('+'), o = 1: a tail ('-'); 0xffffffff = none.
int euler_unitig_links(euler_ctx *ctx, const char *text, const uint64_t *off, uint64_t n, uint32_t K, uint32_t *links)
{
    ENTER(ctx);
    if (n && (!text || !off || !links)) return euler_fail(ctx, EULER_ERR_ARG, "null argument");
    if (K < 2 || K > 63) return euler_fail(ctx, EULER_ERR_ARG, "K %u out of range [2,63]", K);
    if (!n) return EULER_OK;
    if (n >= 0xfffffffeull) return euler_fail(ctx, EULER_ERR_RANGE, "too many contigs");
    const u64 B = off[n];
    DevTmp<char> d_text(ctx, B + 16);
    DevTmp<u64> d_off(ctx, n + 1);
    DevTmp<u32> d_links(ctx, 16 * n);
    TMP_CHECK(ctx, d_text); TMP_CHECK(ctx, d_off); TMP_CHECK(ctx, d_links);
    EULER_TRY(upload(ctx, d_text, text, B));
    EULER_TRY(upload(ctx, d_off, (const u64 *)off, n + 1));
    // the 64-bit end tables use the all-ones word as EMPTY, which is the poly-T 32-mer: K >= 32 takes 128-bit tables
    if (K >= 32) EULER_TRY(wide_unitig_link_graph(ctx, d_text, d_off, n, K, d_links));
    else EULER_TRY(unitig_link_graph(ctx, d_text, d_off, n, K, d_links));
    EULER_TRY(download(ctx, links, d_links.get(), 16 * n));
    FINISH(ctx);
}

int euler_hash_build(euler_ctx *ctx, const uint64_t *keys, const uint32_t *values, uint64_t n, uint64_t capacity,
                     uint64_t *TK, uint32_t *TV)
{
    ENTER(ctx);
    if (!TK || !TV || capacity == 0 || capacity < n) return euler_fail(ctx, EULER_ERR_ARG, "bad table arguments");
    DevTmp<u64> dk(ctx, n), dTK(ctx, capacity), flags(ctx, 1);
    DevTmp<u32> dv(ctx, n), dTV(ctx, capacity);
    TMP_CHECK(ctx, dTK); TMP_CHECK(ctx, dTV); TMP_CHECK(ctx, flags);
    EULER_TRY(upload(ctx, dk, (const u64 *)keys, n));
    EULER_TRY(upload(ctx, dv, values, n));
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(graph_plain_build(ctx, dk, dv, n, dTK, dTV, capacity, flags));
    EULER_TRY(download(ctx, (u64 *)TK, dTK.get(), capacity));
    EULER_TRY(download(ctx, TV, dTV.get(), capacity));
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "hash table full");
    return EULER_OK;
}

int euler_hash_lookup(euler_ctx *ctx, const uint64_t *TK, const uint32_t *TV, uint64_t capacity, const uint64_t *queries,
                      uint64_t nq, uint32_t *out)
{
    ENTER(ctx);
    if (!nq) return EULER_OK;
    if (!TK || !TV || !capacity || !out) return euler_fail(ctx, EULER_ERR_ARG, "bad table arguments");
    DevTmp<u64> dTK(ctx, capacity), dq(ctx, nq);
    DevTmp<u32> dTV(ctx, capacity), dout(ctx, nq);
    TMP_CHECK(ctx, dout);
    EULER_TRY(upload(ctx, dTK, (const u64 *)TK, capacity));
    EULER_TRY(upload(ctx, dTV, TV, capacity));
    EULER_TRY(upload(ctx, dq, (const u64 *)queries, nq));
    PlainTable pt = {dTK, dTV, capacity};
    EULER_TRY(graph_plain_lookup(ctx, pt, dq, nq, dout));
    EULER_TRY(download(ctx, out, dout.get(), nq));
    FINISH(ctx);
}

int euler_exclusive_scan_u32(euler_ctx *ctx, const uint32_t *in, uint64_t n, uint32_t *out)
{
    ENTER(ctx);
    if (!n) return EULER_OK;
    DevTmp<u32> d(ctx, n), o(ctx, n);
    TMP_CHECK(ctx, o);
    EULER_TRY(upload(ctx, d, in, n));
    EULER_TRY(scan_exclusive(ctx, ScanInU32{d.get()}, n, o.get(), (u64 *)nullptr));
    EULER_TRY(download(ctx, out, o.get(), n));
    FINISH(ctx);
}

int euler_debruijn_count(euler_ctx *ctx, const uint64_t *lmer_keys, const uint32_t *lmer_values, uint64_t lmer_count,
                         const uint64_t *TK, const uint32_t *TV, uint64_t capacity, uint32_t l, uint64_t vertex_count,
                         uint32_t *lcount, uint32_t *ecount)
{
    ENTER(ctx);
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l out of range");
    if (!lcount || !ecount) return euler_fail(ctx, EULER_ERR_ARG, "null output");
    DevTmp<u64> dk(ctx, lmer_count), dTK(ctx, capacity);
    DevTmp<u32> dv(ctx, lmer_count), dTV(ctx, capacity), dl(ctx, 4 * vertex_count + 4), de(ctx, 4 * vertex_count + 4);
    TMP_CHECK(ctx, dl); TMP_CHECK(ctx, de);
    EULER_TRY(upload(ctx, dk, (const u64 *)lmer_keys, lmer_count));
    EULER_TRY(upload(ctx, dv, lmer_values, lmer_count));
    EULER_TRY(upload(ctx, dTK, (const u64 *)TK, capacity));
    EULER_TRY(upload(ctx, dTV, TV, capacity));
    CUDA_TRY(ctx, cudaMemsetAsync(dl, 0, (4 * vertex_count + 4) * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(de, 0, (4 * vertex_count + 4) * 4, ctx->stream));
    PlainTable pt = {dTK, dTV, capacity};
    EULER_TRY(graph_degree_slots_plain(ctx, dk, dv, lmer_count, l, pt, vertex_count, dl, de));
    EULER_TRY(download(ctx, lcount, dl.get(), 4 * vertex_count));
    EULER_TRY(download(ctx, ecount, de.get(), 4 * vertex_count));
    FINISH(ctx);
}

int euler_setup_vertices(euler_ctx *ctx, const uint64_t *kmer_keys, uint64_t kmer_count, const uint64_t *TK,
                         const uint32_t *TV, uint64_t capacity, const uint32_t *lcount, const uint32_t *lstart,
                         const uint32_t *ecount, const uint32_t *estart, euler_vertex *ev)
{
    ENTER(ctx);
    if (!kmer_count) return EULER_OK;
    if (!ev) return euler_fail(ctx, EULER_ERR_ARG, "null output");
    const u64 n4 = 4 * kmer_count;
    DevTmp<u64> dk(ctx, kmer_count), dTK(ctx, capacity);
    DevTmp<u32> dTV(ctx, capacity), dlc(ctx, n4), dls(ctx, n4), dec(ctx, n4), des(ctx, n4);
    DevTmp<euler_vertex> dev(ctx, kmer_count);
    TMP_CHECK(ctx, dev);
    EULER_TRY(upload(ctx, dk, (const u64 *)kmer_keys, kmer_count));
    EULER_TRY(upload(ctx, dTK, (const u64 *)TK, capacity));
    EULER_TRY(upload(ctx, dTV, TV, capacity));
    EULER_TRY(upload(ctx, dlc, lcount, n4)); EULER_TRY(upload(ctx, dls, lstart, n4));
    EULER_TRY(upload(ctx, dec, ecount, n4)); EULER_TRY(upload(ctx, des, estart, n4));
    CUDA_TRY(ctx, cudaMemsetAsync(dev, 0, kmer_count * sizeof(euler_vertex), ctx->stream));
    PlainTable pt = {dTK, dTV, capacity};
    EULER_TRY(graph_setup_vertices_plain(ctx, dk, kmer_count, pt, kmer_count, dlc, dls, dec, des, dev));
    EULER_TRY(download(ctx, ev, dev.get(), kmer_count));
    FINISH(ctx);
}

int euler_setup_edges(euler_ctx *ctx, const uint64_t *lmer_keys, const uint32_t *lmer_values, const uint32_t *lmer_offsets,
                      uint64_t lmer_count, const uint64_t *TK, const uint32_t *TV, uint64_t capacity, uint32_t l,
                      const uint32_t *lstart, const uint32_t *estart, uint64_t edge_count, euler_edge *ee, uint32_t *lev,
                      uint32_t *ent)
{
    ENTER(ctx);
    if (l < 2 || l > 32) return euler_fail(ctx, EULER_ERR_ARG, "l out of range");
    if (edge_count >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "edge count exceeds u32");
    if (!edge_count || !lmer_count) return EULER_OK;
    // vertex count is not passed by the reference wrapper: lstart/estart are indexed up to the largest id seen in TV
    u64 nv = 0;
    for (u64 i = 0; i < capacity; i++) if (TV[i] != 0xffffffffu && (u64)TV[i] + 1 > nv) nv = (u64)TV[i] + 1;
    const u64 n4 = 4 * nv;
    DevTmp<u64> dk(ctx, lmer_count), dTK(ctx, capacity);
    DevTmp<u32> dv(ctx, lmer_count), dof(ctx, lmer_count), dTV(ctx, capacity), dls(ctx, n4), des(ctx, n4);
    DevTmp<euler_edge> dee(ctx, edge_count);
    DevTmp<u32> dl(ctx, edge_count), de(ctx, edge_count);
    TMP_CHECK(ctx, dee); TMP_CHECK(ctx, dl); TMP_CHECK(ctx, de);
    EULER_TRY(upload(ctx, dk, (const u64 *)lmer_keys, lmer_count));
    EULER_TRY(upload(ctx, dv, lmer_values, lmer_count));
    EULER_TRY(upload(ctx, dof, lmer_offsets, lmer_count));
    EULER_TRY(upload(ctx, dTK, (const u64 *)TK, capacity));
    EULER_TRY(upload(ctx, dTV, TV, capacity));
    EULER_TRY(upload(ctx, dls, lstart, n4)); EULER_TRY(upload(ctx, des, estart, n4));
    CUDA_TRY(ctx, cudaMemsetAsync(dee, 0, edge_count * sizeof(euler_edge), ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(dl, 0, edge_count * 4, ctx->stream));
    CUDA_TRY(ctx, cudaMemsetAsync(de, 0, edge_count * 4, ctx->stream));
    PlainTable pt = {dTK, dTV, capacity};
    EULER_TRY(graph_setup_edges_plain(ctx, dk, dv, dof, lmer_count, l, pt, dls, des, (u32)edge_count, dee, dl, de));
    EULER_TRY(download(ctx, ee, dee.get(), edge_count));
    EULER_TRY(download(ctx, lev, dl.get(), edge_count));
    EULER_TRY(download(ctx, ent, de.get(), edge_count));
    FINISH(ctx);
}

int euler_assign_successor(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *lev, const uint32_t *ent, uint32_t vcount,
                           euler_edge *ee, uint32_t ecount)
{
    ENTER(ctx);
    if (!ecount || !vcount) return EULER_OK;
    DevTmp<euler_vertex> dev(ctx, vcount);
    DevTmp<u32> dl(ctx, ecount), de(ctx, ecount);
    DevTmp<euler_edge> dee(ctx, ecount);
    EULER_TRY(upload(ctx, dev, ev, vcount));
    EULER_TRY(upload(ctx, dl, lev, ecount));
    EULER_TRY(upload(ctx, de, ent, ecount));
    EULER_TRY(upload(ctx, dee, (const euler_edge *)ee, ecount));
    EULER_TRY(tour_assign_successor(ctx, dev, dl, de, vcount, dee, ecount));
    EULER_TRY(download(ctx, ee, dee.get(), ecount));
    FINISH(ctx);
}

int euler_successor_graph(euler_ctx *ctx, const euler_edge *ee, uint32_t ecount, euler_succ_vertex *v)
{
    ENTER(ctx);
    if (!ecount) return EULER_OK;
    DevTmp<euler_edge> dee(ctx, ecount);
    DevTmp<euler_succ_vertex> dv(ctx, ecount);
    TMP_CHECK(ctx, dv);
    EULER_TRY(upload(ctx, dee, ee, ecount));
    EULER_TRY(tour_successor_graph(ctx, dee, ecount, dv));
    EULER_TRY(download(ctx, v, dv.get(), ecount));
    FINISH(ctx);
}

int euler_find_components(euler_ctx *ctx, const euler_succ_vertex *v, uint32_t n, uint32_t *D)
{
    ENTER(ctx);
    if (!n) return EULER_OK;
    DevTmp<euler_succ_vertex> dv(ctx, n);
    DevTmp<u32> dD(ctx, n);
    TMP_CHECK(ctx, dD);
    EULER_TRY(upload(ctx, dv, v, n));
    EULER_TRY(tour_components(ctx, dv, n, dD));
    EULER_TRY(download(ctx, D, dD.get(), n));
    FINISH(ctx);
}

int euler_circuit_vertices(euler_ctx *ctx, const uint32_t *D, uint32_t ecount, uint32_t *C, uint32_t *offset, uint32_t *cv,
                           uint32_t *count)
{
    ENTER(ctx);
    if (!count) return euler_fail(ctx, EULER_ERR_ARG, "null count");
    *count = 0;
    if (!ecount) return EULER_OK;
    DevTmp<u32> dD(ctx, ecount), dC(ctx, ecount), doff(ctx, ecount), dcv(ctx, ecount);
    DevTmp<u64> dcount(ctx, 1);
    TMP_CHECK(ctx, dC); TMP_CHECK(ctx, doff); TMP_CHECK(ctx, dcv); TMP_CHECK(ctx, dcount);
    EULER_TRY(upload(ctx, dD, D, ecount));
    EULER_TRY(tour_circuit_vertices(ctx, dD, ecount, dC, doff, dcv, dcount));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, dcount, &n));
    *count = (u32)n;
    EULER_TRY(download(ctx, C, dC.get(), ecount));
    EULER_TRY(download(ctx, offset, doff.get(), ecount));
    EULER_TRY(download(ctx, cv, dcv.get(), n));
    FINISH(ctx);
}

int euler_circuit_edges(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *ent, uint32_t vcount, const uint32_t *D,
                        const uint32_t *cmap, uint32_t ecount, euler_circuit_edge *out, uint64_t *count)
{
    ENTER(ctx);
    if (!count) return euler_fail(ctx, EULER_ERR_ARG, "null count");
    const u64 cap = *count;
    *count = 0;
    if (!ecount || !vcount) return EULER_OK;
    DevTmp<euler_vertex> dev(ctx, vcount);
    DevTmp<u32> de(ctx, ecount), dD(ctx, ecount), dmap(ctx, ecount);
    EULER_TRY(upload(ctx, dev, ev, vcount));
    EULER_TRY(upload(ctx, de, ent, ecount));
    EULER_TRY(upload(ctx, dD, D, ecount));
    EULER_TRY(upload(ctx, dmap, cmap, ecount));
    euler_circuit_edge *d_out = nullptr;
    u64 n = 0;
    EULER_TRY(tour_circuit_edges(ctx, dev, nullptr, de, vcount, dD, dmap, ecount, &d_out, &n));
    *count = n;
    if (out) {
        if (cap < n) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small");
        EULER_TRY(download(ctx, out, (const euler_circuit_edge *)d_out, n));
    }
    FINISH(ctx);
}

int euler_spanning_forest(euler_ctx *ctx, const euler_circuit_edge *cg, uint64_t cg_count, uint32_t cg_vcount, uint32_t *tree,
                          uint32_t *tree_count)
{
    ENTER(ctx);
    if (!tree_count) return euler_fail(ctx, EULER_ERR_ARG, "null count");
    *tree_count = 0;
    if (!cg_count || !cg_vcount) return EULER_OK;
    DevTmp<euler_circuit_edge> dcg(ctx, cg_count);
    DevTmp<u32> dtree(ctx, cg_count);
    TMP_CHECK(ctx, dtree);
    EULER_TRY(upload(ctx, dcg, cg, cg_count));
    u32 nt = 0;
    EULER_TRY(tour_spanning_forest(ctx, dcg, cg_count, cg_vcount, dtree, &nt));
    *tree_count = nt;
    EULER_TRY(download(ctx, tree, dtree.get(), nt));
    FINISH(ctx);
}

int euler_mark_spanning(euler_ctx *ctx, const euler_circuit_edge *cg, uint64_t cg_count, const uint32_t *tree,
                        uint32_t tree_count, uint32_t ecount, uint32_t *mark)
{
    ENTER(ctx);
    if (!ecount) return EULER_OK;
    DevTmp<euler_circuit_edge> dcg(ctx, cg_count);
    DevTmp<u32> dtree(ctx, tree_count), dmark(ctx, ecount);
    TMP_CHECK(ctx, dmark);
    EULER_TRY(upload(ctx, dcg, cg, cg_count));
    EULER_TRY(upload(ctx, dtree, tree, tree_count));
    EULER_TRY(tour_mark_spanning(ctx, dcg, dtree, tree_count, ecount, dmark));
    EULER_TRY(download(ctx, mark, dmark.get(), ecount));
    FINISH(ctx);
}

int euler_swipe(euler_ctx *ctx, const euler_vertex *ev, const uint32_t *ent, uint32_t vcount, euler_edge *ee,
                const uint32_t *mark, uint32_t ecount)
{
    ENTER(ctx);
    if (!ecount || !vcount) return EULER_OK;
    DevTmp<euler_vertex> dev(ctx, vcount);
    DevTmp<u32> de(ctx, ecount), dmark(ctx, ecount);
    DevTmp<euler_edge> dee(ctx, ecount);
    EULER_TRY(upload(ctx, dev, ev, vcount));
    EULER_TRY(upload(ctx, de, ent, ecount));
    EULER_TRY(upload(ctx, dmark, mark, ecount));
    EULER_TRY(upload(ctx, dee, (const euler_edge *)ee, ecount));
    EULER_TRY(tour_swipe(ctx, dev, de, vcount, dee, dmark, ecount));
    EULER_TRY(download(ctx, ee, dee.get(), ecount));
    FINISH(ctx);
}

int euler_contig_starts(euler_ctx *ctx, const euler_edge *ee, uint32_t ecount, uint32_t *start)
{
    ENTER(ctx);
    if (!ecount) return EULER_OK;
    DevTmp<euler_edge> dee(ctx, ecount);
    DevTmp<u32> ds(ctx, ecount);
    TMP_CHECK(ctx, ds);
    EULER_TRY(upload(ctx, dee, ee, ecount));
    EULER_TRY(tour_contig_starts(ctx, dee, ecount, ds));
    EULER_TRY(download(ctx, start, ds.get(), ecount));
    FINISH(ctx);
}

int euler_emit_contigs(euler_ctx *ctx, const euler_vertex *ev, uint32_t vcount, const euler_edge *ee, uint32_t ecount,
                       uint32_t l, char *out, uint64_t *out_bytes, uint64_t *ncontigs)
{
    ENTER(ctx);
    if (!out_bytes || !ncontigs) return euler_fail(ctx, EULER_ERR_ARG, "null size pointers");
    if (l < 2 || l > 33) return euler_fail(ctx, EULER_ERR_ARG, "l out of range");
    const u64 cap = *out_bytes;
    *out_bytes = 0; *ncontigs = 0;
    if (!ecount || !vcount) return EULER_OK;
    DevTmp<euler_vertex> dev(ctx, vcount);
    DevTmp<euler_edge> dee(ctx, ecount);
    EULER_TRY(upload(ctx, dev, ev, vcount));
    EULER_TRY(upload(ctx, dee, ee, ecount));
    char *d_text = nullptr;
    u64 bytes = 0, nc = 0;
    EULER_TRY(tour_emit_contigs(ctx, dev, vcount, dee, ecount, l, &d_text, &bytes, &nc));
    *out_bytes = bytes; *ncontigs = nc;
    if (out) {
        if (cap < bytes) return euler_fail(ctx, EULER_ERR_ARG, "output capacity too small");
        EULER_TRY(download(ctx, out, (const char *)d_text, bytes));
    }
    FINISH(ctx);
}

}  // extern "C"
