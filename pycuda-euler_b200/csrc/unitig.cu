// unitig.cu -- unitig ("compacted de Bruijn") contigs of the reference CPU assembler on device:
// referenceAssembler.build (:25-42) + get_contig_forward (:59-77) + all_contigs (:79-88), for K = 2..63.
//
// Nodes are the both-strand K-mers whose count exceeds `limit` (a palindrome counts 2n).  This file describes their
// graph once, as clean.cu takes it: the node ids of the four forward extensions of every node, its twin and its
// both-strand count.  clean.cu applies the link rule, optionally cleans the graph up, and spells every unitig once.
//
// The stage is written once for both key widths.  One-word keys (u64) live in common.cuh's table, two-word keys
// (K128, {lo, hi}) in wide.cuh's; the overloads below are all that differs.  Both tables use the all-ones key as
// EMPTY.  Unitigs and dictionaries store canonical K-mers, and the canonical form of the poly-T 32-mer is poly-A, so
// one word serves up to K = 32.  The link graph stores contig ends as they are, poly-T included, so it uses one word
// up to K = 31 only.  No K-mer of K <= 63 bases is all ones in two words, which is why every job stops at K = 63.
#include "kernels.h"
#include "scan.cuh"
#include "tmp.cuh"
#include "wide.cuh"

#define UB 256

// ---- key-width primitives ----------------------------------------------------------------------------------------
__device__ __forceinline__ bool operator==(K128 a, K128 b) { return eq128(a, b); }
__device__ __forceinline__ bool operator<(K128 a, K128 b) { return lt128(a, b); }
__device__ __forceinline__ bool is_empty(u64 x) { return x == EULER_EMPTY_KEY; }
__device__ __forceinline__ bool is_empty(K128 x) { return is_empty128(x); }
__device__ __forceinline__ u64 revcomp(u64 x, u32 K) { return revcomp64(x, K); }
__device__ __forceinline__ K128 revcomp(K128 x, u32 K) { return revcomp128(x, K); }
// x followed by base `code`; push_base keeps the last K bases of that
__device__ __forceinline__ u64 shl_base(u64 x, u32 code) { return (x << 2) | code; }
__device__ __forceinline__ K128 shl_base(K128 x, u32 code) { return shl2_or(x, code); }
__device__ __forceinline__ u64 push_base(u64 x, u32 code, u32 K) { return shl_base(x, code) & key_mask_d(K); }
__device__ __forceinline__ K128 push_base(K128 x, u32 code, u32 K) { return and128(shl2_or(x, code), mask128(K)); }
// K-mer i of a dictionary given as low and high words (hi is not read for one-word keys)
template <typename Key> __device__ Key dict_key(const u64 *lo, const u64 *hi, u64 i, u32 K);
template <> __device__ __forceinline__ u64 dict_key<u64>(const u64 *lo, const u64 *, u64 i, u32 K) { return lo[i] & key_mask_d(K); }
template <> __device__ __forceinline__ K128 dict_key<K128>(const u64 *lo, const u64 *hi, u64 i, u32 K)
{
    return and128(K128{lo[i], hi[i]}, mask128(K));
}
__device__ __forceinline__ u64 key_find(const u64 *keys, u64 cap, u64 x) { return table_find(keys, cap, x); }
__device__ __forceinline__ u64 key_find(const K128 *keys, u64 cap, K128 x) { return wide_find(keys, cap, x); }
__device__ __forceinline__ u64 key_insert(u64 *keys, u64 cap, u64 x) { return table_insert(keys, cap, x, cap / EULER_BUCKET); }
__device__ __forceinline__ u64 key_insert(K128 *keys, u64 cap, K128 x) { return wide_insert(keys, cap, x, (u32)(cap / WIDE_BUCKET)); }
static int key_table_clear(euler_ctx *ctx, u64 *keys, u32 *vals, u64 cap) { return graph_table_clear(ctx, keys, vals, cap); }
static int key_table_clear(euler_ctx *ctx, K128 *keys, u32 *vals, u64 cap) { return wide_table_clear(ctx, keys, vals, cap); }
// canonical K-mer counts of the reads; d_stats[2] |= 1 on table overflow
static int key_count(euler_ctx *ctx, const void *d_buf, u64 B, const u32 *d_bits, u32 K, u64 *keys, u32 *cnt, u64 cap, u64 *d_stats)
{
    return enc_count_canonical(ctx, d_buf, B, d_bits, K, keys, cnt, cap, TableHash{0, 0}, d_stats);
}
static int key_count(euler_ctx *ctx, const void *d_buf, u64 B, const u32 *d_bits, u32 K, K128 *keys, u32 *cnt, u64 cap, u64 *d_stats)
{
    return wide_count_tiled(ctx, d_buf, B, d_bits, K, keys, cnt, cap, d_stats);
}

// ---- the node graph ---------------------------------------------------------------------------------------------
// strands of slot i that are nodes: 0, 1 (a palindrome) or 2
template <typename Key>
struct NodeWeight {
    const Key *keys;
    const u32 *cnt;
    u32 K, limit;
    __device__ __forceinline__ u32 operator()(u64 i) const
    {
        const Key c = keys[i];
        if (is_empty(c)) return 0u;
        const u32 v = cnt[i];   // loaded ahead of the palindrome test: the two-word instance spills more otherwise
        const bool pal = c == revcomp(c, K);
        const u32 n = pal ? 2u * v : v;
        if (n <= limit) return 0u;
        return pal ? 1u : 2u;
    }
};

// node id of K-mer x if present (count > limit) else EULER_NO_ID
template <typename Key>
__device__ __forceinline__ u32 node_of(const Key *keys, const u32 *cnt, const u32 *base, u64 cap, u32 K, u32 limit, Key x)
{
    const Key r = revcomp(x, K);
    const bool fwd = !(r < x);
    const u64 slot = key_find(keys, cap, fwd ? x : r);
    if (slot == EULER_NO_SLOT) return EULER_NO_ID;
    const u32 n = x == r ? 2u * cnt[slot] : cnt[slot];
    if (n <= limit) return EULER_NO_ID;
    return base[slot] + (fwd ? 0u : 1u);
}

template <typename Key>
__global__ void __launch_bounds__(UB) unitig_nodes_kernel(const Key *__restrict__ keys, const u32 *__restrict__ cnt,
                                                          const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                          Key *__restrict__ nkeys)
{
    const u64 slot = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= cap) return;
    const Key c = keys[slot];
    if (is_empty(c)) return;
    const Key r = revcomp(c, K);
    const bool pal = c == r;
    if ((pal ? 2u * cnt[slot] : cnt[slot]) <= limit) return;
    nkeys[base[slot]] = c;
    if (!pal) nkeys[base[slot] + 1] = r;
}

// clean.cu's view of the node graph: the node ids of the four forward extensions and the twin, and (ncnt != NULL) the
// both-strand count
template <typename Key>
__global__ void __launch_bounds__(UB) unitig_nbr_kernel(const Key *__restrict__ keys, const u32 *__restrict__ cnt,
                                                        const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                        const Key *__restrict__ nkeys, u32 n, u32 *__restrict__ nbr,
                                                        u32 *__restrict__ twin_id, u32 *__restrict__ ncnt)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Key x = nkeys[i];
    const Key tw = revcomp(x, K);
    twin_id[i] = node_of(keys, cnt, base, cap, K, limit, tw);
    for (u32 b = 0; b < 4; b++) nbr[4ull * i + b] = node_of(keys, cnt, base, cap, K, limit, push_base(x, b, K));
    if (!ncnt) return;
    const u64 slot = key_find(keys, cap, tw < x ? tw : x);
    ncnt[i] = x == tw ? 2u * cnt[slot] : cnt[slot];
}

// count table (canonical K-mers, SoA) -> unitig text in ctx->text_buf.  cp == NULL: plain unitigs; else after the
// graph clean-up of clean.cu, with h_sums (may be NULL) the per-contig count sums
template <typename Key>
static int unitigs_from_table(euler_ctx *ctx, const Key *keys, const u32 *cnt, u64 cap, u32 K, u32 limit,
                              const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                              u64 sums_cap, euler_clean_stats *st, UnitigsKept *keep = nullptr)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0; *st = euler_clean_stats{};
    DevTmp<u32> base(ctx, cap);
    DevTmp<u64> total(ctx, 1);
    TMP_CHECK(ctx, base); TMP_CHECK(ctx, total);
    EULER_TRY(scan_exclusive(ctx, NodeWeight<Key>{keys, cnt, K, limit}, cap, base.get(), total.get()));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, total, &n));
    if (!n) return EULER_OK;
    if (n >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "unitig node count exceeds u32");
    const euler_clean_params p = cp ? *cp : euler_clean_params{};   // plain unitigs: no round
    const bool counts = p.max_rounds || h_sums || keep;
    DevTmp<Key> nkeys(ctx, n);
    DevTmp<u32> nbr(ctx, 4 * n), twin_id(ctx, n), ncnt(ctx, counts ? n : 0);
    TMP_CHECK(ctx, nkeys); TMP_CHECK(ctx, nbr); TMP_CHECK(ctx, twin_id); TMP_CHECK(ctx, ncnt);
    unitig_nodes_kernel<<<grid_for(cap, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys.get());
    unitig_nbr_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys.get(), (u32)n, nbr, twin_id,
                                                                counts ? ncnt.get() : nullptr);
    CUDA_TRY(ctx, cudaGetLastError());
    return clean_unitigs(ctx, (u32)n, K, (const u64 *)nkeys.get(), sizeof(Key) / sizeof(u64), nbr, twin_id,
                         counts ? ncnt.get() : nullptr, p, d_out, out_bytes, ncontigs, h_sums, sums_cap, st, keep);
}

template <typename Key>
static int unitigs_from_reads_w(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, u32 K, u32 limit,
                                const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                                u64 sums_cap, euler_clean_stats *st)
{
    const u64 cap = euler_hash_capacity(B);
    DevTmp<u64> d_stats(ctx, 8);
    DevTmp<u32> d_bits(ctx, B / 32 + 2), tc(ctx, cap);
    DevTmp<Key> tk(ctx, cap);
    TMP_CHECK(ctx, d_bits); TMP_CHECK(ctx, d_stats); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc);
    EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, 8 * sizeof(u64), ctx->stream));
    EULER_TRY(key_table_clear(ctx, tk.get(), tc, cap));
    EULER_TRY(key_count(ctx, d_buf, B, d_bits, K, tk.get(), tc, cap, d_stats));
    u64 h[3];
    EULER_TRY(read_u64s(ctx, d_stats, h, 3));
    if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
    return unitigs_from_table(ctx, tk.get(), tc.get(), cap, K, limit, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
}

int unitigs_from_reads(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, u32 K, u32 limit,
                       const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                       euler_clean_stats *st)
{
    if (K <= 32)
        return unitigs_from_reads_w<u64>(ctx, d_buf, d_off, nreads, B, K, limit, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
    return unitigs_from_reads_w<K128>(ctx, d_buf, d_off, nreads, B, K, limit, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
}

// ---- a K-mer dictionary as input (referenceAssembler.all_contigs(d, k) takes the dict of build()) -------
template <typename Key>
__global__ void __launch_bounds__(UB) kmer_dict_insert_kernel(const u64 *__restrict__ lo, const u64 *__restrict__ hi,
                                                               const u32 *__restrict__ counts, u64 n, u32 K, Key *__restrict__ tk,
                                                               u32 *__restrict__ tc, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Key x = dict_key<Key>(lo, hi, i, K), r = revcomp(x, K);
    const u64 slot = key_insert(tk, cap, x < r ? x : r);
    if (slot == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    // the table stores the canonical count n with both-strand count n (2n for a palindrome, :31-35)
    const u32 v = counts[i];
    atomicMax(tc + slot, x == r ? (v + 1u) / 2u : v);
}
int unitig_dict_table(euler_ctx *ctx, const u64 *d_keys, const u32 *d_counts, u64 n, u32 K, u64 *tk, u32 *tc, u64 cap, u64 *d_flags)
{
    if (!n) return EULER_OK;
    kmer_dict_insert_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_keys, nullptr, d_counts, n, K, tk, tc, cap, d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    return EULER_OK;
}

// after kmer_dict_insert_kernel: flag 2 when a key's count is not the both-strand count the table now gives it (an
// odd count on a palindrome, or a key and its twin given with different counts)
template <typename Key>
__global__ void __launch_bounds__(UB) kmer_dict_check_kernel(const u64 *__restrict__ lo, const u64 *__restrict__ hi,
                                                              const u32 *__restrict__ counts, u64 n, u32 K,
                                                              const Key *__restrict__ tk, const u32 *__restrict__ tc, u64 cap,
                                                              u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const Key x = dict_key<Key>(lo, hi, i, K), r = revcomp(x, K);
    const u64 slot = key_find(tk, cap, x < r ? x : r);
    if (slot == EULER_NO_SLOT) return;   // the insert has flagged a full table
    const u32 v = counts[i];
    const bool pal = x == r;
    if ((pal && (v & 1u)) || (pal ? 2u * tc[slot] : tc[slot]) != v) atomicOr((unsigned long long *)flags, 2ull);
}

template <typename Key>
static int unitigs_from_dict_w(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K,
                               const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                               u64 sums_cap, euler_clean_stats *st)
{
    const u64 cap = euler_hash_capacity(n);
    DevTmp<Key> tk(ctx, cap);
    DevTmp<u32> tc(ctx, cap);
    DevTmp<u64> flags(ctx, 1);
    TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc); TMP_CHECK(ctx, flags);
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(key_table_clear(ctx, tk.get(), tc, cap));
    kmer_dict_insert_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_lo, d_hi, d_counts, n, K, tk.get(), tc.get(), cap, flags.get());
    if (cp) kmer_dict_check_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_lo, d_hi, d_counts, n, K, tk.get(), tc.get(), cap, flags.get());
    CUDA_TRY(ctx, cudaGetLastError());
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f & 1) return euler_fail(ctx, EULER_ERR_OVERFLOW, "K-mer table full");
    if (f & 2) return euler_fail(ctx, EULER_ERR_ARG, "K-mer counts are not both-strand counts (an odd count on a palindrome, "
                                                     "or a key and its reverse complement with different counts)");
    return unitigs_from_table(ctx, tk.get(), tc.get(), cap, K, 0, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
}

int unitigs_from_dict(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K,
                      const euler_clean_params *cp, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                      euler_clean_stats *st)
{
    if (K <= 32) return unitigs_from_dict_w<u64>(ctx, d_lo, d_hi, d_counts, n, K, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
    return unitigs_from_dict_w<K128>(ctx, d_lo, d_hi, d_counts, n, K, cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
}

// ---- link graph of the contigs: referenceAssembler.all_contigs :90-111 ------------------------------------
// heads[x[:k]] = (i,'+'), tails[twin(x[-k:])] = (i,'-') (a later contig overwrites an earlier one: max i);
// G[i][0] = for y in fw(x[-k:]): heads hit, tails hit; G[i][1] = for z in fw(twin(x[:k])): heads hit, tails hit.
template <typename Key>
__device__ __forceinline__ Key encode_text_kmer(const char *s, u32 K)
{
    Key x{};
    for (u32 i = 0; i < K; i++) {
        const unsigned char c = (unsigned char)s[i];
        x = shl_base(x, ((c >> 1) ^ (c >> 2)) & 3u);
    }
    return x;
}
template <typename Key>
__global__ void __launch_bounds__(UB) contig_ends_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n, u32 K,
                                                          Key *__restrict__ hk, u32 *__restrict__ hv, Key *__restrict__ tk,
                                                          u32 *__restrict__ tv, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const Key head = encode_text_kmer<Key>(text + b, K);
    const Key tail = revcomp(encode_text_kmer<Key>(text + e - K, K), K);
    const u64 sh = key_insert(hk, cap, head), st = key_insert(tk, cap, tail);
    if (sh == EULER_NO_SLOT || st == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    atomicMax(hv + sh, (u32)i + 1u);
    atomicMax(tv + st, (u32)i + 1u);
}
template <typename Key>
__global__ void __launch_bounds__(UB) contig_links_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n, u32 K,
                                                           const Key *__restrict__ hk, const u32 *__restrict__ hv,
                                                           const Key *__restrict__ tk, const u32 *__restrict__ tv, u64 cap,
                                                           u32 *__restrict__ links)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 *out = links + 16 * i;
    for (int j = 0; j < 16; j++) out[j] = EULER_NO_ID;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const Key last = encode_text_kmer<Key>(text + e - K, K);
    const Key first_tw = revcomp(encode_text_kmer<Key>(text + b, K), K);
    for (int side = 0; side < 2; side++) {
        const Key x = side ? first_tw : last;
        for (u32 c = 0; c < 4; c++) {
            const Key y = push_base(x, c, K);
            const u64 sh = key_find(hk, cap, y), st = key_find(tk, cap, y);
            if (sh != EULER_NO_SLOT) out[8 * side + 2 * c] = hv[sh] - 1u;
            if (st != EULER_NO_SLOT) out[8 * side + 2 * c + 1] = tv[st] - 1u;
        }
    }
}
template <typename Key>
static int link_graph_w(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links)
{
    const u64 cap = ((u64)((double)(n < 16 ? 16 : n) / 0.55) + 1 + 1023) / 1024 * 1024;
    DevTmp<Key> hk(ctx, cap), tk(ctx, cap);
    DevTmp<u32> hv(ctx, cap), tv(ctx, cap);
    DevTmp<u64> flags(ctx, 1);
    TMP_CHECK(ctx, hk); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, hv); TMP_CHECK(ctx, tv); TMP_CHECK(ctx, flags);
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(key_table_clear(ctx, hk.get(), hv, cap));
    EULER_TRY(key_table_clear(ctx, tk.get(), tv, cap));
    contig_ends_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_text, d_off, n, K, hk.get(), hv.get(), tk.get(), tv.get(), cap, flags.get());
    contig_links_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_text, d_off, n, K, hk.get(), hv.get(), tk.get(), tv.get(), cap, d_links);
    CUDA_TRY(ctx, cudaGetLastError());
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "contig end table full");
    return EULER_OK;
}

int unitig_link_graph(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links)
{
    if (!n) return EULER_OK;
    if (K <= 31) return link_graph_w<u64>(ctx, d_text, d_off, n, K, d_links);
    return link_graph_w<K128>(ctx, d_text, d_off, n, K, d_links);
}

// ---- multi-k: the contigs of step i - 1 raise the counts of step i (rule in euler_b200.h) -----------------------
__device__ __forceinline__ u64 rc_push(u64 r, u32 code, u32 K) { return (r >> 2) | ((u64)(3u - code) << (2 * (K - 1))); }
__device__ __forceinline__ K128 rc_push(K128 r, u32 code, u32 K) { return shr2_or_top(r, 3u - code, 2 * (K - 1)); }
__device__ __forceinline__ u32 text_code(const char *s, u64 i)
{
    const unsigned char c = (unsigned char)s[i];
    return ((c >> 1) ^ (c >> 2)) & 3u;
}

#define MK_RUN 64   // window starts per thread

// Every K-window of the previous step's contigs (text, off[nc + 1] with '\n' terminators, count sums, contigs from
// n_starts on are cycles written on Kp-mers): count = max(count, w_C) with w_C = max(limit + 1, sum / L_C), ceil(w / 2)
// on a palindrome.  A thread covers MK_RUN consecutive text positions, rolling both strands through each contig's run.
// A cycle of L_C K-mers is read as its cyclic sequence text[0, L_C) from its start, so it gives all L_C rotations.
// stats[2] |= 1 on a full table; stats[4] += canonical K-mers whose count crosses limit here.
template <typename Key>
__global__ void __launch_bounds__(UB) multik_contig_kmers_kernel(const char *__restrict__ text, const u64 *__restrict__ off,
                                                                  const u64 *__restrict__ sums, u64 nc, u64 n_starts, u32 Kp,
                                                                  u32 K, u32 limit, Key *__restrict__ tk, u32 *__restrict__ tc,
                                                                  u64 cap, u64 *__restrict__ stats)
{
    const u64 p0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * MK_RUN;
    const u64 bytes = off[nc];
    if (p0 >= bytes) return;
    const u64 p1 = p0 + MK_RUN < bytes ? p0 + MK_RUN : bytes;
    u64 lo = 0, hi = nc;   // the contig holding p0: the last c with off[c] <= p0
    while (hi - lo > 1) {
        const u64 mid = (lo + hi) / 2;
        if (off[mid] <= p0) lo = mid; else hi = mid;
    }
    u64 added = 0;
    bool full = false;
    for (u64 c = lo; c < nc && off[c] < p1; c++) {
        const u64 b = off[c], n = off[c + 1] - b - 1, L = n - Kp + 1;   // bases, Kp-mers
        if (n < K) continue;
        const bool cyc = c >= n_starts;
        const u64 s = p0 > b ? p0 - b : 0, e0 = cyc ? L : n - K + 1, e = p1 - b < e0 ? p1 - b : e0;   // window starts [s, e)
        if (s >= e) continue;
        const u64 wm = sums[c] / L;
        const u32 w = (u32)(wm > (u64)limit + 1 ? (wm < 0xffffffffull ? wm : 0xffffffffull) : (u64)limit + 1);
        Key x{}, r{};
        for (u64 j = s; j < s + K - 1; j++) {
            const u32 code = text_code(text + b, j < n ? j : j % L);
            x = shl_base(x, code);
            r = rc_push(r, code, K);
        }
        for (u64 i = s; i < e; i++) {
            const u64 j = i + K - 1;
            const u32 code = text_code(text + b, j < n ? j : j % L);
            x = push_base(x, code, K);
            r = rc_push(r, code, K);
            const bool pal = x == r;
            const u64 slot = key_insert(tk, cap, r < x ? r : x);
            if (slot == EULER_NO_SLOT) { full = true; continue; }
            const u32 v = pal ? (u32)(((u64)w + 1u) / 2u) : w;   // in u64: w may be 0xffffffff
            const u32 old = atomicMax(tc + slot, v);
            // counts only grow, so exactly one update takes a K-mer from <= limit to > limit
            if ((pal ? 2ull * old : old) <= limit && (pal ? 2ull * v : v) > limit) added++;
        }
    }
    if (added) atomicAdd((unsigned long long *)(stats + 4), (unsigned long long)added);
    if (full) atomicOr((unsigned long long *)(stats + 2), 1ull);
}

// one step: the count table of the reads at K, raised by the previous contigs (prev_nc of them, Kp-mers, on the device
// in ctx->text_buf and prev), then clean_unitigs.  keep: where this step's contigs stay for the next one.
template <typename Key>
static int multik_step_w(euler_ctx *ctx, const void *d_buf, u64 B, const u32 *d_bits, u32 K, u32 Kp, u32 limit,
                         const euler_clean_params &cp, const UnitigsKept &prev, u64 prev_nc, u64 prev_bytes, UnitigsKept *keep,
                         char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap, euler_clean_stats *st,
                         u64 *nodes_added)
{
    const u64 cap = euler_hash_capacity(B + prev_bytes);
    DevTmp<u64> d_stats(ctx, 8);
    DevTmp<u32> tc(ctx, cap);
    DevTmp<Key> tk(ctx, cap);
    TMP_CHECK(ctx, d_stats); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, tc);
    CUDA_TRY(ctx, cudaMemsetAsync(d_stats, 0, 8 * sizeof(u64), ctx->stream));
    EULER_TRY(key_table_clear(ctx, tk.get(), tc, cap));
    if (B) EULER_TRY(key_count(ctx, d_buf, B, d_bits, K, tk.get(), tc, cap, d_stats));
    if (prev_nc) {
        multik_contig_kmers_kernel<Key><<<grid_for((prev_bytes + MK_RUN - 1) / MK_RUN, UB), UB, 0, ctx->stream>>>(
            (const char *)ctx->text_buf.p, prev.off.ptr(), prev.sums.ptr(), prev_nc, prev.n_starts, Kp, K, limit, tk.get(), tc.get(),
            cap, d_stats.get());
        CUDA_TRY(ctx, cudaGetLastError());
    }
    u64 h[5];
    EULER_TRY(read_u64s(ctx, d_stats, h, 5));
    if (h[2]) return euler_fail(ctx, EULER_ERR_OVERFLOW, "count table overflow");
    *nodes_added = h[4];
    return unitigs_from_table(ctx, tk.get(), tc.get(), cap, K, limit, &cp, d_out, out_bytes, ncontigs, h_sums, sums_cap, st, keep);
}

int unitigs_multik(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u64 B, const u32 *ks, u32 nk, u32 limit,
                   const euler_clean_params *params, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums, u64 sums_cap,
                   euler_multik_step *steps)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0;
    DevTmp<u32> d_bits(ctx, B / 32 + 2);
    TMP_CHECK(ctx, d_bits);
    if (B) EULER_TRY(enc_mark_starts(ctx, d_off, nreads, B, d_bits));
    UnitigsKept kept;   // offsets and sums of the previous step; its text is ctx->text_buf until this step spells
    u64 nc = 0, bytes = 0;
    int rc = EULER_OK;
    for (u32 i = 0; i < nk && rc == EULER_OK; i++) {
        const bool last = i + 1 == nk;
        const u32 K = ks[i], Kp = i ? ks[i - 1] : 0;
        char *text = nullptr;
        u64 nb = 0, n = 0, added = 0;
        euler_clean_stats st{};
        if (K <= 32)
            rc = multik_step_w<u64>(ctx, d_buf, B, d_bits, K, Kp, limit, params[i], kept, nc, bytes, last ? nullptr : &kept, &text,
                                    &nb, &n, last ? h_sums : nullptr, sums_cap, &st, &added);
        else
            rc = multik_step_w<K128>(ctx, d_buf, B, d_bits, K, Kp, limit, params[i], kept, nc, bytes, last ? nullptr : &kept, &text,
                                     &nb, &n, last ? h_sums : nullptr, sums_cap, &st, &added);
        nc = n; bytes = nb;
        if (steps) steps[i] = euler_multik_step{K, n, nb - n, added, st};
        if (last) { *d_out = text; *out_bytes = nb; *ncontigs = n; }
    }
    return rc;
}
