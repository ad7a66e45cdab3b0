// wide.cuh -- two-word (128-bit) key arithmetic and the open-addressing table over them.
// A len-mer (len <= 64) is packed MSB-first in the low 2*len bits of {hi, lo}, the same convention
// as the 64-bit path (pyencode.py:42-67) and oracle_impl.h's 128-bit instantiation.
#pragma once
#include "common.cuh"

struct __align__(16) K128 {
    u64 lo, hi;
};

__device__ __forceinline__ bool eq128(K128 a, K128 b) { return a.lo == b.lo && a.hi == b.hi; }
__device__ __forceinline__ bool lt128(K128 a, K128 b) { return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo); }
__device__ __forceinline__ bool is_empty128(K128 a) { return (a.lo & a.hi) == ~0ull; }
__device__ __forceinline__ K128 and128(K128 a, K128 b) { return K128{a.lo & b.lo, a.hi & b.hi}; }
__device__ __forceinline__ K128 mask128(u32 len)
{
    if (len >= 64) return K128{~0ull, ~0ull};
    if (len >= 32) return K128{~0ull, len == 32 ? 0ull : ((1ull << (2 * (len - 32))) - 1ull)};
    return K128{(1ull << (2 * len)) - 1ull, 0ull};
}
__device__ __forceinline__ K128 shr128(K128 a, u32 s)   // 0 <= s < 128
{
    if (s == 0) return a;
    if (s >= 64) return K128{a.hi >> (s - 64), 0ull};
    return K128{(a.lo >> s) | (a.hi << (64 - s)), a.hi >> s};
}
__device__ __forceinline__ K128 shl2_or(K128 a, u32 code) { return K128{(a.lo << 2) | code, (a.hi << 2) | (a.lo >> 62)}; }
// rolling reverse complement: drop the lowest base, put `code` at bit position `top` (= 2*(len-1))
__device__ __forceinline__ K128 shr2_or_top(K128 a, u32 code, u32 top)
{
    K128 r{(a.lo >> 2) | (a.hi << 62), a.hi >> 2};
    if (top >= 64) r.hi |= (u64)code << (top - 64);
    else r.lo |= (u64)code << top;
    return r;
}
__device__ __forceinline__ u64 revcomp64_full(u64 x)
{
    u64 y = __brevll(~x);
    return ((y >> 1) & 0x5555555555555555ull) | ((y & 0x5555555555555555ull) << 1);
}
__device__ __forceinline__ K128 revcomp128(K128 x, u32 len)
{
    const K128 full{revcomp64_full(x.hi), revcomp64_full(x.lo)};   // 64-base reverse complement
    return shr128(full, 128 - 2 * len);
}
__device__ __forceinline__ K128 canon128(K128 x, u32 len)
{
    const K128 r = revcomp128(x, len);
    return lt128(r, x) ? r : x;
}
// code of base i (0 = first / most significant) of a len-mer
__device__ __forceinline__ u32 base_at(K128 x, u32 len, u32 i) { return (u32)(shr128(x, 2 * (len - 1 - i)).lo & 3ull); }

// ---- table: buckets of two 16-byte keys (one 32 B sector) -----------------------------------------
#define WIDE_BUCKET 2
__device__ __forceinline__ u64 wide_hash_bucket(K128 key, u32 nbuckets)
{
    const u64 x = key.lo ^ (key.hi * 0xC2B2AE3D27D4EB4Full) ^ (key.hi >> 31);
    const u64 h = (x ^ (x >> 29)) * 0x9E3779B97F4A7C15ull;
    return ((h >> 32) * (u64)nbuckets) >> 32;
}
__device__ __forceinline__ K128 ld_k128_cg(const K128 *p)
{
    K128 r;
    asm volatile("ld.global.cg.v2.b64 {%0,%1}, [%2];" : "=l"(r.lo), "=l"(r.hi) : "l"(p));
    return r;
}
__device__ __forceinline__ K128 cas128(K128 *addr, K128 cmp, K128 val)
{
    K128 old;
    asm volatile(
        "{\n\t.reg .b128 c, v, o;\n\tmov.b128 c, {%2, %3};\n\tmov.b128 v, {%4, %5};\n\t"
        "atom.global.cas.b128 o, [%6], c, v;\n\tmov.b128 {%0, %1}, o;\n\t}"
        : "=l"(old.lo), "=l"(old.hi)
        : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(addr)
        : "memory");
    return old;
}
// slot of `key` after inserting it if absent; EULER_NO_SLOT when max_probe buckets were all full
__device__ __forceinline__ u64 wide_insert(K128 *keys, u64 cap, K128 key, u32 max_probe)
{
    const u32 nb = (u32)(cap / WIDE_BUCKET);
    const K128 empty{~0ull, ~0ull};
    u64 b = wide_hash_bucket(key, nb);
    for (u32 probe = 0; probe < max_probe; probe++) {
#pragma unroll
        for (int j = 0; j < WIDE_BUCKET; j++) {
            K128 *p = keys + b * WIDE_BUCKET + j;
            K128 cur = ld_k128_cg(p);
            if (is_empty128(cur)) cur = cas128(p, empty, key);
            if (is_empty128(cur) || eq128(cur, key)) return b * WIDE_BUCKET + j;
        }
        if (++b == nb) b = 0;
    }
    return EULER_NO_SLOT;
}
__device__ __forceinline__ u64 wide_find(const K128 *keys, u64 cap, K128 key)
{
    const u32 nb = (u32)(cap / WIDE_BUCKET);
    u64 b = wide_hash_bucket(key, nb);
    for (u32 probe = 0; probe < nb; probe++) {
#pragma unroll
        for (int j = 0; j < WIDE_BUCKET; j++) {
            const K128 cur = ld_k128_cg(keys + b * WIDE_BUCKET + j);
            if (eq128(cur, key)) return b * WIDE_BUCKET + j;
            if (is_empty128(cur)) return EULER_NO_SLOT;
        }
        if (++b == nb) b = 0;
    }
    return EULER_NO_SLOT;
}

// One probe step for `key` at bucket b (two 16-byte slots = one 32-byte sector, loaded with a single 256-bit
// load): slot index of the key after claiming it if absent, EULER_NO_SLOT when both slots hold other keys.
// *fresh is incremented when this call claimed the slot.
__device__ __forceinline__ u64 wide_probe_step(K128 *keys, u64 b, K128 key, u32 &fresh)
{
    K128 *bk = keys + b * WIDE_BUCKET;
    const K4 q = ld_bucket_cg((const u64 *)bk);
    const bool m0 = q.k[0] == key.lo && q.k[1] == key.hi, m1 = q.k[2] == key.lo && q.k[3] == key.hi;
    if (m0 | m1) return b * WIDE_BUCKET + (m0 ? 0 : 1);
    const bool e0 = (q.k[0] & q.k[1]) == ~0ull, e1 = (q.k[2] & q.k[3]) == ~0ull;
    const K128 empty{~0ull, ~0ull};
    for (int j = e0 ? 0 : (e1 ? 1 : 2); j < WIDE_BUCKET; j++) {   // a lost race moves on to the next slot through its own CAS
        const K128 old = cas128(bk + j, empty, key);
        if (is_empty128(old)) { fresh++; return b * WIDE_BUCKET + j; }
        if (eq128(old, key)) return b * WIDE_BUCKET + j;
    }
    return EULER_NO_SLOT;
}

// ---- wide.cu launchers (asynchronous on ctx->stream) -----------------------------------------------
// d_stats: [0] += forward l-windows, [1] += forward (l-1)-windows, [2] |= 1 on table overflow
int wide_count(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u32 l, K128 *keys, u32 *cnt, u64 cap, u64 *d_stats);
// tiled form (warp per 28 chunks, shared-memory compaction of the valid keys); d_bits = read-start bitmap
int wide_count_tiled(euler_ctx *ctx, const void *d_buf, u64 n_bases, const u32 *d_bits, u32 l, K128 *keys, u32 *cnt, u64 cap,
                     u64 *d_stats);
int wide_table_clear(euler_ctx *ctx, K128 *keys, u32 *vals, u64 cap);
int wide_vertex_insert(euler_ctx *ctx, const K128 *lt_keys, u64 lt_cap, u32 l, K128 *vt_keys, u64 vt_cap, u64 *d_flags);
int wide_slot_scan(euler_ctx *ctx, const K128 *keys, u64 cap, u32 len, u32 *d_base, u64 *d_total);
int wide_compact_vertices(euler_ctx *ctx, const K128 *vt_keys, const u32 *vt_base, u64 vt_cap, u32 k, u64 *vk_lo, u64 *vk_hi);
int wide_compact_lmers(euler_ctx *ctx, const K128 *lt_keys, const u32 *lt_cnt, const u32 *lt_base, u64 lt_cap, u32 l, u64 *lk_lo,
                       u64 *lk_hi, u32 *lvals);
// ascending (hi, lo) order on bits [0, nbits); vals (may be NULL) follow their keys
int wide_sort(euler_ctx *ctx, u64 *lo, u64 *hi, u32 *vals, u64 n, int nbits);
int wide_assign_sorted_ids(euler_ctx *ctx, const u64 *vk_lo, const u64 *vk_hi, u64 nv, const K128 *vt_keys, u64 vt_cap, u32 k,
                           u32 *id0, u32 *id1);
// tf[i] = (last base code) | (first base code << 2) of l-mer i, consumed by graph_setup_edges
int wide_degree_slots(euler_ctx *ctx, const u64 *lk_lo, const u64 *lk_hi, const u32 *lvals, u64 nl, u32 l, const K128 *vt_keys,
                      const u32 *id0, const u32 *id1, u64 vt_cap, u32 *lcount, u32 *ecount, u32 *ev1, u32 *ev2, unsigned char *tf);

// ---- wide_unitig.cu (unitig stage, K = 33..63; link graph, K = 32..63)
int wide_unitig_from_table(euler_ctx *ctx, const K128 *keys, const u32 *cnt, u64 cap, u32 K, u32 limit, char **d_out,
                           u64 *out_bytes, u64 *ncontigs, u64 *n_nodes);
// canonical count table from a both-strand K-mer dictionary (keys as lo / hi words, counts)
int wide_unitig_dict_table(euler_ctx *ctx, const u64 *d_lo, const u64 *d_hi, const u32 *d_counts, u64 n, u32 K, K128 *tk, u32 *tc,
                           u64 cap, u64 *d_flags);
// links[16 i + 8 side + 2 base + (0 head '+' | 1 tail '-')] of n contigs (text without separators, off[n+1])
int wide_unitig_link_graph(euler_ctx *ctx, const char *d_text, const u64 *d_off, u64 n, u32 K, u32 *d_links);
// (key, count) filter: keep count > limit, compact
int wide_filter_counts(euler_ctx *ctx, const u64 *lo, const u64 *hi, const u32 *vals, u64 n, u32 limit, u32 *d_base, u64 *out_lo,
                       u64 *out_hi, u32 *out_vals, u64 *d_total);

// ---- wide_dist.cu (k-mer-space partition over 16-byte keys)
int wide_dist_scatter(euler_ctx *ctx, const void *d_buf, const u64 *d_off, u64 nreads, u32 l, u32 nranks, u64 *d_counts,
                      u64 *d_cursors, void *d_send, const u64 *d_seg_off, u64 seg_cap);
int wide_count_keys(euler_ctx *ctx, const void *d_keys, u64 n, K128 *keys, u32 *cnt, u64 cap, u64 *d_stats);
int wide_own_flags(euler_ctx *ctx, const K128 *keys, u64 cap, u32 l, u32 rank, u32 nranks, unsigned char *own);
int wide_dist_vertex_insert(euler_ctx *ctx, const K128 *lt_keys, u64 lt_cap, u32 l, const unsigned char *own, K128 *vt_keys,
                            u64 vt_cap, u64 *d_flags);
int wide_homed_scan(euler_ctx *ctx, const K128 *keys, const unsigned char *own, u64 cap, u32 l, u32 *d_base, u64 *d_total);
int wide_compact_homed(euler_ctx *ctx, const K128 *lt_keys, const u32 *lt_cnt, const unsigned char *own, const u32 *base, u64 cap,
                       u32 l, u64 *lk_lo, u64 *lk_hi, u32 *lvals);
int wide_foreign_in_edges(euler_ctx *ctx, const K128 *lt_keys, const u32 *lt_cnt, const unsigned char *own, u64 cap, u32 l,
                          const K128 *vt_keys, const u32 *id0, u64 vt_cap, u32 *ecount);
