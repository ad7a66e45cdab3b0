// unitig.cu -- unitig ("compacted de Bruijn") contigs of the reference CPU assembler on device:
// referenceAssembler.build (:25-42) + get_contig_forward (:59-77) + all_contigs (:79-88).
//
// Nodes are the both-strand K-mers whose count exceeds `limit`.  A link x -> y exists iff y is the
// only present forward extension of x, x is the only present backward extension of y, and y is not
// twin(x) (hairpin stop, :70-71).  The components of that link graph are simple paths and cycles,
// i.e. the unitigs; chain.cuh ranks and spells them.  Every unitig exists on both strands; it is
// written once (the component whose label is not larger than its reverse-complement component's).
#include "chain.cuh"
#include "kernels.h"
#include "scan.cuh"
#include "tmp.cuh"

#define UB 256

__device__ __forceinline__ u64 canon_k(u64 x, u32 K)
{
    const u64 r = revcomp64(x, K);
    return x < r ? x : r;
}

// both-strand count of the K-mer stored canonically at `slot`
__device__ __forceinline__ u32 both_count(const u64 *keys, const u32 *cnt, u64 slot, u32 K)
{
    const u64 c = keys[slot];
    const u32 n = cnt[slot];
    return c == revcomp64(c, K) ? 2u * n : n;
}

struct NodeWeight {
    const u64 *keys;
    const u32 *cnt;
    u32 K, limit;
    __device__ __forceinline__ u32 operator()(u64 i) const
    {
        const u64 c = keys[i];
        if (c == EULER_EMPTY_KEY) return 0u;
        const bool pal = c == revcomp64(c, K);
        const u32 n = pal ? 2u * cnt[i] : cnt[i];
        if (n <= limit) return 0u;
        return pal ? 1u : 2u;
    }
};

// node id of K-mer x if present (count > limit) else EULER_NO_ID
__device__ __forceinline__ u32 node_of(const u64 *keys, const u32 *cnt, const u32 *base, u64 cap, u32 K, u32 limit, u64 x)
{
    const u64 r = revcomp64(x, K);
    const u64 c = x < r ? x : r;
    const u64 slot = table_find(keys, cap, c);
    if (slot == EULER_NO_SLOT) return EULER_NO_ID;
    const u32 n = (c == r && c == x) ? 2u * cnt[slot] : cnt[slot];
    if (n <= limit) return EULER_NO_ID;
    return base[slot] + (x == c ? 0u : 1u);
}

__global__ void __launch_bounds__(UB) unitig_nodes_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                          const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                          u64 *__restrict__ nkeys)
{
    const u64 slot = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= cap) return;
    const u64 c = keys[slot];
    if (c == EULER_EMPTY_KEY) return;
    if (both_count(keys, cnt, slot, K) <= limit) return;
    const u64 r = revcomp64(c, K);
    nkeys[base[slot]] = c;
    if (c != r) nkeys[base[slot] + 1] = r;
}

// referenceAssembler.get_contig_forward :59-77, one step, for every node
__global__ void __launch_bounds__(UB) unitig_links_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                          const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                          const u64 *__restrict__ nkeys, u32 n, u32 *__restrict__ succ,
                                                          u32 *__restrict__ twin_id)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 x = nkeys[i];
    const u64 mask = key_mask_d(K);
    const u64 tw = revcomp64(x, K);
    twin_id[i] = node_of(keys, cnt, base, cap, K, limit, tw);
    u32 s = n;
    u32 nf = 0, cand_id = EULER_NO_ID;
    u64 cand = 0;
    for (u32 b = 0; b < 4; b++) {  // fw(): km[1:] + x
        const u64 y = ((x << 2) | b) & mask;
        const u32 id = node_of(keys, cnt, base, cap, K, limit, y);
        if (id != EULER_NO_ID) { nf++; cand = y; cand_id = id; }
    }
    if (nf == 1 && cand != tw) {
        u32 nb = 0;
        for (u32 b = 0; b < 4; b++) {  // bw(): x + km[:-1]
            const u64 z = ((u64)b << (2 * (K - 1))) | (cand >> 2);
            if (node_of(keys, cnt, base, cap, K, limit, z) != EULER_NO_ID) nb++;
        }
        if (nb == 1) s = cand_id;
    }
    succ[i] = s;
}

struct UnitigChainModel {
    const u64 *nkeys;
    const u32 *succ_;
    const u32 *twin_id;
    static constexpr u32 HEAD_APPENDS = 0;
    __device__ __forceinline__ u32 succ(u32 i) const { return succ_[i]; }
    __device__ __forceinline__ u64 head_key(u32 i) const { return nkeys[i]; }
    __device__ __forceinline__ u64 head_key_hi(u32) const { return 0ull; }
    __device__ __forceinline__ char base(u32 i) const { return "ACGT"[nkeys[i] & 3]; }
    // write each unitig once: the strand whose component label is the smaller one
    __device__ __forceinline__ bool emit(const u32 *D, u32 i) const { return D[i] <= D[twin_id[i]]; }
};

// count table (canonical K-mers, SoA) -> unitig text in ctx->text_buf
int unitig_from_table(euler_ctx *ctx, const u64 *keys, const u32 *cnt, u64 cap, u32 K, u32 limit, char **d_out,
                      u64 *out_bytes, u64 *ncontigs, u64 *n_nodes)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0; *n_nodes = 0;
    DevTmp<u32> base(ctx, cap);
    DevTmp<u64> total(ctx, 1);
    TMP_CHECK(ctx, base); TMP_CHECK(ctx, total);
    EULER_TRY(scan_exclusive(ctx, NodeWeight{keys, cnt, K, limit}, cap, base.get(), total.get()));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, total, &n));
    *n_nodes = n;
    if (!n) return EULER_OK;
    if (n >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "unitig node count exceeds u32");
    DevTmp<u64> nkeys(ctx, n);
    DevTmp<u32> succ(ctx, n), twin_id(ctx, n);
    TMP_CHECK(ctx, nkeys); TMP_CHECK(ctx, succ); TMP_CHECK(ctx, twin_id);
    unitig_nodes_kernel<<<grid_for(cap, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys);
    unitig_links_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys, (u32)n, succ, twin_id);
    CUDA_TRY(ctx, cudaGetLastError());
    UnitigChainModel m = {nkeys, succ, twin_id};
    return chain_emit(ctx, m, (u32)n, K, d_out, out_bytes, ncontigs);
}

// clean.cu's view of the node graph: the node ids of the four forward extensions, the twin and the both-strand count
__global__ void __launch_bounds__(UB) unitig_nbr_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ cnt,
                                                        const u32 *__restrict__ base, u64 cap, u32 K, u32 limit,
                                                        const u64 *__restrict__ nkeys, u32 n, u32 *__restrict__ nbr,
                                                        u32 *__restrict__ twin_id, u32 *__restrict__ ncnt)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 x = nkeys[i];
    const u64 mask = key_mask_d(K);
    twin_id[i] = node_of(keys, cnt, base, cap, K, limit, revcomp64(x, K));
    for (u32 b = 0; b < 4; b++) nbr[4ull * i + b] = node_of(keys, cnt, base, cap, K, limit, ((x << 2) | b) & mask);
    ncnt[i] = both_count(keys, cnt, table_find(keys, cap, canon_k(x, K)), K);
}

// unitig_from_table after the graph clean-up of clean.cu; h_sums (may be NULL): per-contig count sums
int unitig_clean_from_table(euler_ctx *ctx, const u64 *keys, const u32 *cnt, u64 cap, u32 K, u32 limit,
                            const euler_clean_params &p, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                            u64 sums_cap, euler_clean_stats *st)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0; *st = euler_clean_stats{};
    DevTmp<u32> base(ctx, cap);
    DevTmp<u64> total(ctx, 1);
    TMP_CHECK(ctx, base); TMP_CHECK(ctx, total);
    EULER_TRY(scan_exclusive(ctx, NodeWeight{keys, cnt, K, limit}, cap, base.get(), total.get()));
    u64 n = 0;
    EULER_TRY(read_u64(ctx, total, &n));
    if (!n) return EULER_OK;
    if (n >= 0xffffffffull) return euler_fail(ctx, EULER_ERR_RANGE, "unitig node count exceeds u32");
    DevTmp<u64> nkeys(ctx, n);
    DevTmp<u32> nbr(ctx, 4 * n), twin_id(ctx, n), ncnt(ctx, n);
    TMP_CHECK(ctx, nkeys); TMP_CHECK(ctx, nbr); TMP_CHECK(ctx, twin_id); TMP_CHECK(ctx, ncnt);
    unitig_nodes_kernel<<<grid_for(cap, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys);
    unitig_nbr_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(keys, cnt, base, cap, K, limit, nkeys, (u32)n, nbr, twin_id, ncnt);
    CUDA_TRY(ctx, cudaGetLastError());
    return clean_unitigs(ctx, (u32)n, K, nkeys, 1, nbr, twin_id, ncnt, p, d_out, out_bytes, ncontigs, h_sums, sums_cap, st);
}

// ---- a K-mer dictionary as input (referenceAssembler.all_contigs(d, k) takes the dict of build()) -------
__global__ void __launch_bounds__(UB) kmer_dict_insert_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ counts, u64 n,
                                                               u32 K, u64 *__restrict__ tk, u32 *__restrict__ tc, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 x = keys[i] & key_mask_d(K), r = revcomp64(x, K);
    const u64 c = x < r ? x : r;
    const u64 slot = table_insert(tk, cap, c, cap / EULER_BUCKET);
    if (slot == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    // the table stores the canonical count n with both-strand count n (2n for a palindrome, :31-35)
    const u32 v = counts[i];
    atomicMax(tc + slot, x == r ? (v + 1u) / 2u : v);
}
int unitig_dict_table(euler_ctx *ctx, const u64 *d_keys, const u32 *d_counts, u64 n, u32 K, u64 *tk, u32 *tc, u64 cap, u64 *d_flags)
{
    if (!n) return EULER_OK;
    kmer_dict_insert_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_keys, d_counts, n, K, tk, tc, cap, d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    return EULER_OK;
}

// after kmer_dict_insert_kernel: flag 2 when a key's count is not the both-strand count the table now gives it (an
// odd count on a palindrome, or a key and its twin given with different counts)
__global__ void __launch_bounds__(UB) kmer_dict_check_kernel(const u64 *__restrict__ keys, const u32 *__restrict__ counts, u64 n,
                                                              u32 K, const u64 *__restrict__ tk, const u32 *__restrict__ tc,
                                                              u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 x = keys[i] & key_mask_d(K), r = revcomp64(x, K);
    const u64 slot = table_find(tk, cap, x < r ? x : r);
    if (slot == EULER_NO_SLOT) return;   // the insert has flagged a full table
    const u32 v = counts[i];
    if ((x == r && (v & 1u)) || both_count(tk, tc, slot, K) != v) atomicOr((unsigned long long *)flags, 2ull);
}
int unitig_dict_check(euler_ctx *ctx, const u64 *d_keys, const u32 *d_counts, u64 n, u32 K, const u64 *tk, const u32 *tc, u64 cap,
                      u64 *d_flags)
{
    if (!n) return EULER_OK;
    kmer_dict_check_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_keys, d_counts, n, K, tk, tc, cap, d_flags);
    CUDA_TRY(ctx, cudaGetLastError());
    return EULER_OK;
}

// ---- link graph of the contigs: referenceAssembler.all_contigs :90-111 ------------------------------------
// heads[x[:k]] = (i,'+'), tails[twin(x[-k:])] = (i,'-') (a later contig overwrites an earlier one: max i);
// G[i][0] = for y in fw(x[-k:]): heads hit, tails hit; G[i][1] = for z in fw(twin(x[:k])): heads hit, tails hit.
__device__ __forceinline__ u64 encode_text_kmer(const char *s, u32 K)
{
    u64 x = 0;
    for (u32 i = 0; i < K; i++) {
        const unsigned char c = (unsigned char)s[i];
        x = (x << 2) | (u64)(((c >> 1) ^ (c >> 2)) & 3u);
    }
    return x;
}
__global__ void __launch_bounds__(UB) contig_ends_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n, u32 K,
                                                          u64 *__restrict__ hk, u32 *__restrict__ hv, u64 *__restrict__ tk,
                                                          u32 *__restrict__ tv, u64 cap, u64 *flags)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const u64 head = encode_text_kmer(text + b, K);
    const u64 tail = revcomp64(encode_text_kmer(text + e - K, K), K);
    const u64 sh = table_insert(hk, cap, head, cap / EULER_BUCKET), st = table_insert(tk, cap, tail, cap / EULER_BUCKET);
    if (sh == EULER_NO_SLOT || st == EULER_NO_SLOT) { atomicOr((unsigned long long *)flags, 1ull); return; }
    atomicMax(hv + sh, (u32)i + 1u);
    atomicMax(tv + st, (u32)i + 1u);
}
__global__ void __launch_bounds__(UB) contig_links_kernel(const char *__restrict__ text, const u64 *__restrict__ off, u64 n, u32 K,
                                                           const u64 *__restrict__ hk, const u32 *__restrict__ hv,
                                                           const u64 *__restrict__ tk, const u32 *__restrict__ tv, u64 cap,
                                                           u32 *__restrict__ links)
{
    const u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 *out = links + 16 * i;
    for (int j = 0; j < 16; j++) out[j] = EULER_NO_ID;
    const u64 b = off[i], e = off[i + 1];
    if (e - b < K) return;
    const u64 mask = key_mask_d(K);
    const u64 last = encode_text_kmer(text + e - K, K);
    const u64 first_tw = revcomp64(encode_text_kmer(text + b, K), K);
    for (int side = 0; side < 2; side++) {
        const u64 x = side ? first_tw : last;
        for (u32 c = 0; c < 4; c++) {
            const u64 y = ((x << 2) | c) & mask;
            const u64 sh = table_find(hk, cap, y), st = table_find(tk, cap, y);
            if (sh != EULER_NO_SLOT) out[8 * side + 2 * c] = hv[sh] - 1u;
            if (st != EULER_NO_SLOT) out[8 * side + 2 * c + 1] = tv[st] - 1u;
        }
    }
}
int unitig_link_graph(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links)
{
    if (!n) return EULER_OK;
    const u64 cap = ((u64)((double)(n < 16 ? 16 : n) / 0.55) + 1 + 1023) / 1024 * 1024;
    DevTmp<u64> hk(ctx, cap), tk(ctx, cap), flags(ctx, 1);
    DevTmp<u32> hv(ctx, cap), tv(ctx, cap);
    TMP_CHECK(ctx, hk); TMP_CHECK(ctx, tk); TMP_CHECK(ctx, hv); TMP_CHECK(ctx, tv); TMP_CHECK(ctx, flags);
    CUDA_TRY(ctx, cudaMemsetAsync(flags, 0, sizeof(u64), ctx->stream));
    EULER_TRY(graph_table_clear(ctx, hk, hv, cap));
    EULER_TRY(graph_table_clear(ctx, tk, tv, cap));
    contig_ends_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_text, d_off, n, K, hk, hv, tk, tv, cap, flags);
    contig_links_kernel<<<grid_for(n, UB), UB, 0, ctx->stream>>>(d_text, d_off, n, K, hk, hv, tk, tv, cap, d_links);
    CUDA_TRY(ctx, cudaGetLastError());
    u64 f = 0;
    EULER_TRY(read_u64(ctx, flags, &f));
    if (f) return euler_fail(ctx, EULER_ERR_OVERFLOW, "contig end table full");
    return EULER_OK;
}
