// common.cuh -- shared device/host helpers for libeuler_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/euler_b200.h"

typedef unsigned long long u64;
typedef unsigned int u32;

#define EULER_EMPTY_KEY 0xFFFFFFFFFFFFFFFFull
#define EULER_NO_ID 0xFFFFFFFFu
#define EULER_SMS 148
#define EULER_PINNED_WORDS 1024

// ---------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------
// Owns its device memory: freed on destruction, so the device it was allocated on must be current then.  Move-only.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept
    {
        if (this != &o) {
            if (p) cudaFree(p);
            p = o.p; cap = o.cap;
            o.p = nullptr; o.cap = 0;
        }
        return *this;
    }
    ~DevBuf() { if (p) cudaFree(p); }
};

struct Pipeline;

struct euler_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    // pinned host staging for small device->host reads
    u64 *h_pinned = nullptr;   // EULER_PINNED_WORDS u64 of pinned host memory for small read-backs
    Pipeline *pipe = nullptr;
    DevBuf scan_state;  // tile descriptors of the single-pass scan
    DevBuf cg_buf;      // circuit edges of the last tour_circuit_edges call
    DevBuf text_buf;    // contig text of the last emission
    u64 text_gen = 0;   // bumped by every emission: a cached text is valid only for the generation it was written in
    cudaEvent_t ev[8] = {};
    int num_sms = EULER_SMS;
    size_t l2_bytes = 0;
    size_t persist_max = 0;   // bytes of L2 that may be set aside for persisting lines
    size_t window_max = 0;    // largest access-policy window
    size_t l2_part_budget = 0;  // table bytes one count pass may own (0 = default)
};

int euler_fail(euler_ctx *ctx, int code, const char *fmt, ...);

#define CUDA_TRY(ctx, expr)                                                                        \
    do {                                                                                           \
        cudaError_t e_ = (expr);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return euler_fail((ctx), EULER_ERR_CUDA, "%s:%d %s: %s", __FILE__, __LINE__, #expr,    \
                              cudaGetErrorString(e_));                                             \
    } while (0)

#define EULER_TRY(expr)                                                                            \
    do {                                                                                           \
        int r_ = (expr);                                                                           \
        if (r_ != EULER_OK) return r_;                                                             \
    } while (0)

// grow-only device buffer
int dev_reserve(euler_ctx *ctx, DevBuf &b, size_t bytes);

template <typename T>
struct DevArr {
    DevBuf b;
    T *ptr() const { return (T *)b.p; }
    int reserve(euler_ctx *ctx, size_t n) { return dev_reserve(ctx, b, (n ? n : 1) * sizeof(T)); }
};

static inline unsigned grid_for(u64 n, unsigned block)
{
    u64 g = (n + block - 1) / block;
    if (g < 1) g = 1;
    if (g > 0x7fffffffull) g = 0x7fffffffull;
    return (unsigned)g;
}

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
#ifdef __CUDACC__

// Table hash: xor-fold, one 64-bit multiply (Fibonacci), then the top 32 bits scaled into the
// bucket range with a single 32x32->64 multiply.  Buckets are 4 consecutive slots (one 32-byte
// sector), so a probe is one 256-bit load.
#define EULER_BUCKET 4
__device__ __forceinline__ u64 hash_bucket(u64 key, u32 nbuckets)
{
    const u64 h = (key ^ (key >> 29)) * 0x9E3779B97F4A7C15ull;
    return ((h >> 32) * (u64)nbuckets) >> 32;
}

__device__ __forceinline__ u64 key_mask_d(u32 len) { return len >= 32 ? ~0ull : ((1ull << (2 * len)) - 1ull); }

// reverse complement of a len-mer packed MSB-first in the low 2*len bits
__device__ __forceinline__ u64 revcomp64(u64 x, u32 len)
{
    u64 y = __brevll(~x);                                                  // reverse all bits of the complement
    y = ((y >> 1) & 0x5555555555555555ull) | ((y & 0x5555555555555555ull) << 1);  // restore bit order inside each base
    return y >> (64 - 2 * len);
}

__device__ __forceinline__ u64 ld_cg_u64(const u64 *p)
{
    u64 v;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ u32 ld_cg_u32(const u32 *p)
{
    u32 v;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
// streaming 128-bit load (read-once input): non-coherent path, no L1 allocation
__device__ __forceinline__ uint4 ld_stream_v4(const uint4 *p)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

// ---- open-addressing table primitives ---------------------------------------------------------
// Bucketised linear probing: a key lives in its home bucket (4 slots = one 32 B sector) or, when
// that is full, in the following buckets.  Slots of a bucket fill in order, so the first EMPTY
// slot ends a lookup.  Canonical l-mers never equal all-ones (canon(T^32)=A^32=0) and k-mers use
// <= 62 bits, so 0xFFFF... is a safe EMPTY for every key this library stores (SURVEY B3).
#define EULER_NO_SLOT 0xFFFFFFFFFFFFFFFFull
struct K4 {
    u64 k[4];
};
__device__ __forceinline__ K4 ld_bucket_cg(const u64 *p)
{
    K4 r;
    asm volatile("ld.global.cg.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(r.k[0]), "=l"(r.k[1]), "=l"(r.k[2]), "=l"(r.k[3]) : "l"(p));
    return r;
}
__device__ __forceinline__ K4 ld_bucket_nc(const u64 *p)
{
    K4 r;
    asm volatile("ld.global.nc.v4.b64 {%0,%1,%2,%3}, [%4];" : "=l"(r.k[0]), "=l"(r.k[1]), "=l"(r.k[2]), "=l"(r.k[3]) : "l"(p));
    return r;
}

// Try to place / find `key` in the bucket `q` loaded from keys + 4*bucket.  Returns the slot
// index inside the bucket (0..3) or -1 when the bucket is full of other keys.
__device__ __forceinline__ int bucket_claim(u64 *bucket_keys, const K4 &q, u64 key)
{
#pragma unroll
    for (int j = 0; j < EULER_BUCKET; j++) {
        const u64 kv = q.k[j];
        if (kv == key) return j;
        if (kv == EULER_EMPTY_KEY) {
            const u64 old = atomicCAS(bucket_keys + j, EULER_EMPTY_KEY, key);
            if (old == EULER_EMPTY_KEY || old == key) return j;
        }
    }
    return -1;
}

// branch-free bucket match (count kernels)
template <int NK>
__device__ __forceinline__ int bucket_match(const K4 &q, u64 key, int &first_empty)
{
    // slot of `key` among the first NK slots of the bucket or -1; first_empty = first EMPTY slot or NK
    unsigned m = 0, e = 0;
#pragma unroll
    for (int t = 0; t < NK; t++) {
        m |= (q.k[t] == key ? 1u : 0u) << t;
        e |= (q.k[t] == EULER_EMPTY_KEY ? 1u : 0u) << t;
    }
    first_empty = e ? (int)__ffs(e) - 1 : NK;
    return m ? (int)__ffs(m) - 1 : -1;
}

// ---- minimizer-ordered homes -------------------------------------------------------------------
// With a plain hash the ~70 l-mers of a read touch ~70 random sectors of a table far larger than
// L2.  Ordering the table by the key's minimizer (smallest scrambled canonical m-mer) sends the
// ~(l-m+1)/2 consecutive l-mers that share a minimizer to the same EULER_SPAN buckets (256 B), and
// sends an l-mer and its prefix / suffix k-mers to corresponding regions of the l-mer and vertex
// tables, so the graph stage walks both tables almost sequentially.  The minimizer is strand
// symmetric (canonical m-mers), so it can be taken from either orientation of the key.
#define EULER_SPAN 8
struct TableHash {
    u32 span_nb;  // nbuckets - EULER_SPAN when minimizer ordering is on, 0 = plain hash
    u32 m;        // minimizer length (<= 16, <= key length)
};
__device__ __forceinline__ u32 mmer_score(u32 canon_m)
{
    const u32 s = canon_m * 2654435761u;
    return s ^ (s >> 15);
}
// scores of the m-mers of `key` (len bases): min over all of them, over all but the last
// (= the prefix (len-1)-mer's minimizer) and over all but the first (= the suffix's)
__device__ __forceinline__ void min_scores(u64 key, u32 len, u32 m, u32 &all, u32 &but_last, u32 &but_first)
{
    const u64 r = revcomp64(key, len);
    const u32 mmask = m >= 16 ? 0xffffffffu : ((1u << (2 * m)) - 1u);
    const u32 n = len - m + 1;
    all = but_last = but_first = 0xffffffffu;
    for (u32 j = 0; j < n; j++) {
        const u32 w = (u32)(key >> (2 * (len - m - j))) & mmask;
        const u32 rw = (u32)(r >> (2 * j)) & mmask;
        const u32 sc = mmer_score(w < rw ? w : rw);
        all = sc < all ? sc : all;
        if (j + 1 < n) but_last = sc < but_last ? sc : but_last;
        if (j > 0) but_first = sc < but_first ? sc : but_first;
    }
}
__device__ __forceinline__ u64 home_from_score(u64 key, u32 score, u32 nb, TableHash th)
{
    if (!th.span_nb) return hash_bucket(key, nb);
    // the minimum of many scores is far from uniform (it hugs 0); the score is a bijection of the
    // m-mer, so re-mixing it (murmur3 fmix32) gives a uniform region that still depends only on the
    // minimizer's identity
    u32 h = score;
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return (((u64)h * th.span_nb) >> 32) + ((key * 0x9E3779B97F4A7C15ull) >> 61);
}
__device__ __forceinline__ u64 table_home(u64 key, u32 len, u32 nb, TableHash th)
{
    if (!th.span_nb) return hash_bucket(key, nb);
    u32 a, b, c;
    min_scores(key, len, th.m, a, b, c);
    return home_from_score(key, a, nb, th);
}

// ---- co-hashed tables ---------------------------------------------------------------------------------
// The graph stage walks the canonical l-mer table in slot order and looks up each l-mer's prefix and
// suffix vertex.  If the l-mer table is hashed by the canonical form of the PREFIX k-mer of the stored
// (canonical) l-mer -- the very value the vertex table hashes -- an l-mer and its prefix vertex sit at
// the same relative position of their tables: the prefix lookups, the prefix-side degree-slot writes
// and half of the vertex inserts become sequential, only the suffix side stays random.  At most four
// canonical l-mers share a home (one bucket).  TableHash{0, EULER_PREFIX_HOME} selects it.
#define EULER_PREFIX_HOME 0xffffffffu
// c = canonical l-mer, r = its reverse complement, kmask = mask of k = l-1 bases
__device__ __forceinline__ u64 prefix_home_key(u64 c, u64 r, u64 kmask, u32 &flip)
{
    const u64 p = c >> 2, rp = r & kmask;   // rc(prefix(c)) = suffix(rc(c))
    flip = rp < p ? 1u : 0u;
    return flip ? rp : p;
}
// A vertex is the canonical prefix of up to two canonical l-mers (its out-edge when that is canonical
// as written, its in-edge when the reverse complement is).  Both in one bucket raises the bucket-load
// variance (count kernel 1.52 -> 1.88 ms); the second kind one bucket up makes ADJACENT buckets
// correlated, which lengthens the overflow cascades (probe rounds +17 %, 1.77 ms).  It therefore goes
// EULER_FLIP_STRIDE buckets up: still the same neighbourhood of the table for the graph stage.
#define EULER_FLIP_STRIDE 37u
__device__ __forceinline__ u32 prefix_home_bucket(u64 c, u64 r, u64 kmask, u32 nbuckets)
{
    u32 flip;
    const u64 hk = prefix_home_key(c, r, kmask, flip);
    u32 b = (u32)hash_bucket(hk, nbuckets) + (flip ? EULER_FLIP_STRIDE : 0u);
    return b >= nbuckets ? b % nbuckets : b;
}

// ---- degree-slot writes of the edge kernels ----------------------------------------------------------
// Reference layout: lcount[4 v + base], ecount[4 v + base] (pydebruijn.py:107-141) -- four scattered
// 4-byte writes into four different sectors per canonical l-mer.  Paired layout (slot-order ids, where
// the two strands of a vertex have adjacent ids): one 32-byte region per vertex id holding
// [lcount(v) | ecount(partner(v))], partner = the other strand (itself for a palindrome).  The two
// prefix-side writes of an l-mer (lcount of prefix(c), ecount of rc(prefix(c))) then share one sector and
// so do the two suffix-side writes; the vertex pass (graph.cu) reads the regions back and writes the
// reference arrays coalesced.
struct DegOut {
    u32 *lcount, *ecount;   // reference layout (used when deg == NULL)
    u32 *deg;               // paired layout: u32[8 V]
};
__device__ __forceinline__ void deg_put_l(const DegOut &d, u32 v, u32 slot, u32 m)
{
    if (d.deg) d.deg[8ull * v + slot] = m;
    else d.lcount[4ull * v + slot] = m;
}
__device__ __forceinline__ void deg_put_e(const DegOut &d, u32 v, u32 partner, u32 slot, u32 m)
{
    if (d.deg) d.deg[8ull * partner + 4u + slot] = m;
    else d.ecount[4ull * v + slot] = m;
}

// returns slot of `key` after inserting it if absent; EULER_NO_SLOT on overflow. cap % 4 == 0.
__device__ __forceinline__ u64 table_insert_at(u64 *keys, u64 cap, u64 key, u64 home, u64 max_probe)
{
    const u32 nb = (u32)(cap / EULER_BUCKET);
    u64 b = home;
    for (u64 probe = 0; probe < max_probe; probe++) {
        u64 *bk = keys + b * EULER_BUCKET;
        const K4 q = ld_bucket_cg(bk);
        const int j = bucket_claim(bk, q, key);
        if (j >= 0) return b * EULER_BUCKET + j;
        if (++b == nb) b = 0;
    }
    return EULER_NO_SLOT;
}

__device__ __forceinline__ u64 table_find_at(const u64 *keys, u64 cap, u64 key, u64 home)
{
    const u32 nb = (u32)(cap / EULER_BUCKET);
    u64 b = home;
    for (u64 probe = 0; probe < nb; probe++) {
        const K4 q = ld_bucket_nc(keys + b * EULER_BUCKET);
#pragma unroll
        for (int j = 0; j < EULER_BUCKET; j++) {
            if (q.k[j] == key) return b * EULER_BUCKET + j;
            if (q.k[j] == EULER_EMPTY_KEY) return EULER_NO_SLOT;
        }
        if (++b == nb) b = 0;
    }
    return EULER_NO_SLOT;
}

// Vertex id lookup through per-bucket id bases: bbase[b] = id of the first strand stored in bucket b
// (the exclusive scan of the strand weights at the bucket's first slot), so the id of slot j is
// bbase[b] + the weights of the j slots before it -- known from the bucket just loaded.  One u32 per
// bucket instead of one per slot: the array is 4x smaller than id0[] and stays in L2, which removes
// one random DRAM sector per lookup.  k = vertex length (palindromes, weight 1, exist only for even k).
__device__ __forceinline__ u32 table_find_id(const u64 *keys, u64 cap, u64 key, u64 home, const u32 *bbase, u32 k)
{
    const u32 nb = (u32)(cap / EULER_BUCKET);
    u64 b = home;
    for (u64 probe = 0; probe < nb; probe++) {
        const K4 q = ld_bucket_nc(keys + b * EULER_BUCKET);
        u32 before = 0;
#pragma unroll
        for (int j = 0; j < EULER_BUCKET; j++) {
            if (q.k[j] == key) return bbase[b] + before;
            if (q.k[j] == EULER_EMPTY_KEY) return EULER_NO_ID;
            before += (!(k & 1u) && q.k[j] == revcomp64(q.k[j], k)) ? 1u : 2u;
        }
        if (++b == nb) b = 0;
    }
    return EULER_NO_ID;
}

// plain-hash forms (module-level gpuhash API, partitioned path)
__device__ __forceinline__ u64 table_insert(u64 *keys, u64 cap, u64 key, u64 max_probe)
{
    return table_insert_at(keys, cap, key, hash_bucket(key, (u32)(cap / EULER_BUCKET)), max_probe);
}
__device__ __forceinline__ u64 table_find(const u64 *keys, u64 cap, u64 key)
{
    return table_find_at(keys, cap, key, hash_bucket(key, (u32)(cap / EULER_BUCKET)));
}

#endif  // __CUDACC__
