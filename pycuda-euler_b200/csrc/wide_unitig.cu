// wide_unitig.cu -- the unitig stage of unitig.cu on two-word (128-bit) K-mer keys, K = 33..63, plus the
// 128-bit forms of the K-mer dictionary input, the contig link graph (K = 32..63) and the filtered K-mer count
// behind referenceAssembler.build at len = 33..64.
//
// Same graph and rules as unitig.cu: nodes are the both-strand K-mers whose count exceeds `limit` (a palindrome
// counts 2n), x -> y iff y is the only present forward extension of x, x the only present backward extension of
// y and y != twin(x); chain.cuh spells each unitig once.  The table is wide.cuh's: canonical key = the smaller
// of the two strands in (hi, lo) order, EMPTY = all ones in both words.  A K-mer of K <= 63 bases has at most
// 62 bits in its high word, so no K-mer equals EMPTY; a 64-mer can (poly-T), which is why unitigs and link
// graphs stop at K = 63 while counting, whose keys are canonical, goes to 64.
#include "chain.cuh"
#include "kernels.h"
#include "scan.cuh"
#include "tmp.cuh"
#include "wide.cuh"

#define WUB 256

// strands of slot i that are nodes: 0, 1 (a palindrome) or 2.  A pass of its own, scanned by the stock u32 scan:
// the shared scan kernel built around a two-word weight functor spills.
__global__ void __launch_bounds__(WUB) wide_node_weight_kernel(const K128 *__restrict__ keys, const u32 *__restrict__ cnt, u64 cap,
                                                                u32 K, u32 limit, u32 *__restrict__ w)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    const K128 c = keys[i];
    u32 v = 0;
    if (!is_empty128(c)) {
        const bool pal = eq128(c, revcomp128(c, K));
        const u32 n = pal ? 2u * cnt[i] : cnt[i];
        if (n > limit) v = pal ? 1u : 2u;
    }
    w[i] = v;
}

// node id of K-mer x if present (count > limit) else EULER_NO_ID
__device__ __forceinline__ u32 wide_node_of(const K128 *keys, const u32 *cnt, const u32 *base, u64 cap, u32 K, u32 limit, K128 x)
{
    const K128 r = revcomp128(x, K);
    const bool fwd = !lt128(r, x);
    const u64 slot = wide_find(keys, cap, fwd ? x : r);
    if (slot == EULER_NO_SLOT) return EULER_NO_ID;
    const u32 n = eq128(x, r) ? 2u * cnt[slot] : cnt[slot];
    if (n <= limit) return EULER_NO_ID;
    return base[slot] + (fwd ? 0u : 1u);
}

__global__ void __launch_bounds__(WUB) wide_unitig_nodes_kernel(const K128 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                                 const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                                 K128 *__restrict__ nkeys)
{
    const u64 slot = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= cap) return;
    const K128 c = keys[slot];
    if (is_empty128(c)) return;
    const K128 r = revcomp128(c, K);
    const bool pal = eq128(c, r);
    if ((pal ? 2u * cnt[slot] : cnt[slot]) <= limit) return;
    nkeys[base[slot]] = c;
    if (!pal) nkeys[base[slot] + 1] = r;
}

// referenceAssembler.get_contig_forward :59-77, one step, for every node
__global__ void __launch_bounds__(WUB) wide_unitig_links_kernel(const K128 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                                 const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                                 const K128 *__restrict__ nkeys, u32 n, u32 *__restrict__ succ,
                                                                 u32 *__restrict__ twin_id)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const K128 x = nkeys[i];
    const K128 mask = mask128(K);
    const K128 tw = revcomp128(x, K);
    twin_id[i] = wide_node_of(keys, cnt, base, cap, K, limit, tw);
    u32 s = n;
    u32 nf = 0, cand_id = EULER_NO_ID;
    K128 cand{0, 0};
    for (u32 b = 0; b < 4; b++) {  // fw(): km[1:] + x
        const K128 y = and128(shl2_or(x, b), mask);
        const u32 id = wide_node_of(keys, cnt, base, cap, K, limit, y);
        if (id != EULER_NO_ID) { nf++; cand = y; cand_id = id; }
    }
    if (nf == 1 && !eq128(cand, tw)) {
        u32 nb = 0;
        for (u32 b = 0; b < 4; b++) {  // bw(): x + km[:-1]
            const K128 z = shr2_or_top(cand, b, 2 * (K - 1));
            if (wide_node_of(keys, cnt, base, cap, K, limit, z) != EULER_NO_ID) nb++;
        }
        if (nb == 1) s = cand_id;
    }
    succ[i] = s;
}

struct WideUnitigChainModel {
    const K128 *nkeys;
    const u32 *succ_;
    const u32 *twin_id;
    static constexpr u32 HEAD_APPENDS = 0;
    __device__ __forceinline__ u32 succ(u32 i) const { return succ_[i]; }
    __device__ __forceinline__ u64 head_key(u32 i) const { return nkeys[i].lo; }
    __device__ __forceinline__ u64 head_key_hi(u32 i) const { return nkeys[i].hi; }
    __device__ __forceinline__ char base(u32 i) const { return "ACGT"[nkeys[i].lo & 3]; }
    // write each unitig once: the strand whose component label is the smaller one
    __device__ __forceinline__ bool emit(const u32 *D, u32 i) const { return D[i] <= D[twin_id[i]]; }
};

int wide_unitig_from_table(euler_ctx *ctx, const K128 *keys, const u32 *cnt, u64 cap, u32 K, u32 limit, char **d_out,
                           u64 *out_bytes, u64 *ncontigs, u64 *n_nodes)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0; *n_nodes = 0;
    DevTmp<u32> weight(ctx, cap), base(ctx, cap);
    DevTmp<u64> total(ctx, 1);
    TMP_CHECK(ctx, weight); TMP_CHECK(ctx, base); TMP_CHECK(ctx, total);
    wide_node_weight_kernel<<<grid_for(cap, WUB), WUB, 0, ctx->stream>>>(keys, cnt, cap, K, limit, weight);
    CUDA_TRY(ctx, cudaGetLastError());
    EULER_TRY(scan_exclusive(ctx, ScanInU32{weight}, cap, base.get(), total.get()));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, total, &n));
    *n_nodes = n;
    if (!n) return EULER_OK;
    if (n >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "unitig node count exceeds u32");
    DevTmp<K128> nkeys(ctx, n);
    DevTmp<u32> succ(ctx, n), twin_id(ctx, n);
    TMP_CHECK(ctx, nkeys); TMP_CHECK(ctx, succ); TMP_CHECK(ctx, twin_id);
    wide_unitig_nodes_kernel<<<grid_for(cap, WUB), WUB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys);
    wide_unitig_links_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys, (u32)n, succ,
                                                                        twin_id);
    CUDA_TRY(ctx, cudaGetLastError());
    WideUnitigChainModel m = {nkeys, succ, twin_id};
    return chain_emit(ctx, m, (u32)n, K, d_out, out_bytes, ncontigs);
}

// clean.cu's view of the node graph, as unitig_nbr_kernel
__global__ void __launch_bounds__(WUB) wide_unitig_nbr_kernel(const K128 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                               const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                               const K128 *__restrict__ nkeys, u32 n, u32 *__restrict__ nbr,
                                                               u32 *__restrict__ twin_id, u32 *__restrict__ ncnt)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const K128 x = nkeys[i];
    const K128 mask = mask128(K);
    const K128 tw = revcomp128(x, K);
    twin_id[i] = wide_node_of(keys, cnt, base, cap, K, limit, tw);
    for (u32 b = 0; b < 4; b++) nbr[4ull * i + b] = wide_node_of(keys, cnt, base, cap, K, limit, and128(shl2_or(x, b), mask));
    const u64 slot = wide_find(keys, cap, lt128(tw, x) ? tw : x);
    ncnt[i] = eq128(x, tw) ? 2u * cnt[slot] : cnt[slot];
}

// wide_unitig_from_table after the graph clean-up of clean.cu
int wide_unitig_clean_from_table(euler_ctx *ctx, const K128 *keys, const u32 *cnt, u64 cap, u32 K, u32 limit,
                                 const euler_clean_params &p, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                                 u64 sums_cap, euler_clean_stats *st)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0; *st = euler_clean_stats{};
    DevTmp<u32> weight(ctx, cap), base(ctx, cap);
    DevTmp<u64> total(ctx, 1);
    TMP_CHECK(ctx, weight); TMP_CHECK(ctx, base); TMP_CHECK(ctx, total);
    wide_node_weight_kernel<<<grid_for(cap, WUB), WUB, 0, ctx->stream>>>(keys, cnt, cap, K, limit, weight);
    CUDA_TRY(ctx, cudaGetLastError());
    EULER_TRY(scan_exclusive(ctx, ScanInU32{weight}, cap, base.get(), total.get()));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, total, &n));
    if (!n) return EULER_OK;
    if (n >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "unitig node count exceeds u32");
    DevTmp<K128> nkeys(ctx, n);
    DevTmp<u32> nbr(ctx, 4 * n), twin_id(ctx, n), ncnt(ctx, n);
    TMP_CHECK(ctx, nkeys); TMP_CHECK(ctx, nbr); TMP_CHECK(ctx, twin_id); TMP_CHECK(ctx, ncnt);
    wide_unitig_nodes_kernel<<<grid_for(cap, WUB), WUB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys);
    wide_unitig_nbr_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys, (u32)n, nbr, twin_id,
                                                                      ncnt);
    CUDA_TRY(ctx, cudaGetLastError());
    return clean_unitigs(ctx, (u32)n, K, (const u64 *)nkeys.get(), 2, nbr, twin_id, ncnt, p, d_out, out_bytes, ncontigs, h_sums,
                         sums_cap, st);
}

// ---- a K-mer dictionary as input (referenceAssembler.all_contigs(d, k) takes the dict of build()) -------
__global__ void __launch_bounds__(WUB) wide_kmer_dict_insert_kernel(const u64 *__restrict__ keys_lo, const u64 *__restrict__ keys_hi,
                                                                     const u32 *__restrict__ counts, u64 n, u32 K,
                                                                     K128 *__restrict__ tk, u32 *__restrict__ tc, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const K128 x = and128(K128{keys_lo[i], keys_hi[i]}, mask128(K)), r = revcomp128(x, K);
    const u64 slot = wide_insert(tk, cap, lt128(r, x) ? r : x, (u32)(cap / WIDE_BUCKET));
    if (slot == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    // the table stores the canonical count n with both-strand count n (2n for a palindrome, :31-35)
    const u32 v = counts[i];
    atomicMax(tc + slot, eq128(x, r) ? (v + 1u) / 2u : v);
}
int wide_unitig_dict_table(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K, K128 *tk, u32 *tc,
                           u64 cap, u64 *d_flags)
{
    if (!n) return EULER_OK;
    wide_kmer_dict_insert_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(d_lo, d_hi, d_counts, n, K, tk, tc, cap, d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    return EULER_OK;
}

// after wide_kmer_dict_insert_kernel: flag 2 as kmer_dict_check_kernel
__global__ void __launch_bounds__(WUB) wide_kmer_dict_check_kernel(const u64 *__restrict__ keys_lo, const u64 *__restrict__ keys_hi,
                                                                    const u32 *__restrict__ counts, u64 n, u32 K,
                                                                    const K128 *__restrict__ tk, const u32 *__restrict__ tc, u64 cap,
                                                                    u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const K128 x = and128(K128{keys_lo[i], keys_hi[i]}, mask128(K)), r = revcomp128(x, K);
    const u64 slot = wide_find(tk, cap, lt128(r, x) ? r : x);
    if (slot == EULER_NO_SLOT) return;   // the insert has flagged a full table
    const u32 v = counts[i];
    const bool pal = eq128(x, r);
    if ((pal && (v & 1u)) || (pal ? 2u * tc[slot] : tc[slot]) != v) atomicOr((unsigned long long *)flags, 2ull);
}
int wide_unitig_dict_check(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K, const K128 *tk,
                           const u32 *tc, u64 cap, u64 *d_flags)
{
    if (!n) return EULER_OK;
    wide_kmer_dict_check_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(d_lo, d_hi, d_counts, n, K, tk, tc, cap, d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    return EULER_OK;
}

// ---- link graph of the contigs (referenceAssembler.all_contigs :90-111), as unitig_link_graph --------------
__device__ __forceinline__ K128 encode_text_kmer128(const char *s, u32 K)
{
    K128 x{0, 0};
    for (u32 i = 0; i < K; i++) {
        const unsigned char c = (unsigned char)s[i];
        x = shl2_or(x, ((c >> 1) ^ (c >> 2)) & 3u);
    }
    return x;
}
__global__ void __launch_bounds__(WUB) wide_contig_ends_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n,
                                                                u32 K, K128 *__restrict__ hk, u32 *__restrict__ hv,
                                                                K128 *__restrict__ tk, u32 *__restrict__ tv, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const K128 head = encode_text_kmer128(text + b, K);
    const K128 tail = revcomp128(encode_text_kmer128(text + e - K, K), K);
    const u32 mp = (u32)(cap / WIDE_BUCKET);
    const u64 sh = wide_insert(hk, cap, head, mp), st = wide_insert(tk, cap, tail, mp);
    if (sh == EULER_NO_SLOT || st == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    atomicMax(hv + sh, (u32)i + 1u);   // a later contig overwrites an earlier one
    atomicMax(tv + st, (u32)i + 1u);
}
__global__ void __launch_bounds__(WUB) wide_contig_links_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n,
                                                                 u32 K, const K128 *__restrict__ hk, const u32 *__restrict__ hv,
                                                                 const K128 *__restrict__ tk, const u32 *__restrict__ tv, u64 cap,
                                                                 u32 *__restrict__ links)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 *out = links + 16 * i;
    for (int j = 0; j < 16; j++) out[j] = EULER_NO_ID;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const K128 mask = mask128(K);
    const K128 last = encode_text_kmer128(text + e - K, K);
    const K128 first_tw = revcomp128(encode_text_kmer128(text + b, K), K);
    for (int side = 0; side < 2; side++) {
        const K128 x = side ? first_tw : last;
        for (u32 c = 0; c < 4; c++) {
            const K128 y = and128(shl2_or(x, c), mask);
            const u64 sh = wide_find(hk, cap, y), st = wide_find(tk, cap, y);
            if (sh != EULER_NO_SLOT) out[8 * side + 2 * c] = hv[sh] - 1u;
            if (st != EULER_NO_SLOT) out[8 * side + 2 * c + 1] = tv[st] - 1u;
        }
    }
}
int wide_unitig_link_graph(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links)
{
    if (!n) return EULER_OK;
    const u64 cap = ((u64)((double)(n < 16 ? 16 : n) / 0.55) + 1 + 1023) / 1024 * 1024;
    DevTmp<K128> hk(ctx, cap), tk(ctx, cap);
    DevTmp<u32> hv(ctx, cap), tv(ctx, cap);
    DevTmp<u64> flags(ctx, 1);
    TMP_CHECK(ctx, hk); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, hv); TMP_CHECK(ctx, tv); TMP_CHECK(ctx, flags);
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(wide_table_clear(ctx, hk, hv, cap));
    EULER_TRY(wide_table_clear(ctx, tk, tv, cap));
    wide_contig_ends_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(d_text, d_off, n, K, hk, hv, tk, tv, cap, flags);
    wide_contig_links_kernel<<<grid_for(n, WUB), WUB, 0, ctx->stream>>>(d_text, d_off, n, K, hk, hv, tk, tv, cap, d_links);
    CUDA_TRY(ctx, cudaGetLastError());
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "contig end table full");
    return EULER_OK;
}

// ---- (key, count) filter over two-word keys: keep count > limit (referenceAssembler.build :37-39) ----------
// graph.cu's one-word filter, once per key word (both passes keep the same entries)
int wide_filter_counts(euler_ctx *ctx, const u64 *lo, const u64 *hi, const u32 *vals, u64 n, u32 limit, u32 *d_base, u64 *out_lo,
                       u64 *out_hi, u32 *out_vals, u64 *d_total)
{
    EULER_TRY(graph_filter_counts(ctx, lo, vals, n, limit, d_base, out_lo, out_vals, d_total));
    return graph_filter_counts(ctx, hi, vals, n, limit, d_base, out_hi, out_vals, d_total);
}
