// chain.cuh -- contig emission for any successor graph whose components are simple paths and
// cycles: predecessor scatter, components, head detection (cycles are cut at their minimum node
// id), pointer-jumping list ranking, contig ordering, length scan and base scatter.
//
// It is the data-parallel form of the reference's host walk generatePartialContig
// (eulercuda.py:351-402): first every chain that has a start node, in ascending start id, then
// every cycle, entered at its smallest node id.  A `Model` supplies what a node spells:
//   n()                       number of nodes
//   succ(i)                   successor node or >= n
//   head_key(i)               k-mer (2-bit packed) that opens a contig headed by node i (head_key_hi: bits 64.. when k > 32)
//   base(i)                   character appended by node i
//   emit(D, i)                whether the component (label array D) of head i is written at all
//   HEAD_APPENDS              1: the head node also appends base(i) (Euler edges)
//                             0: the head node only contributes its k-mer (unitig k-mers)
#pragma once
#include "kernels.h"
#include "scan.cuh"
#include "tmp.cuh"

#define CH_TB 256

template <typename M>
__global__ void __launch_bounds__(CH_TB) ch_pred_kernel(M m, u32 n, u32 *__restrict__ pred)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u32 s = m.succ(t);
    if (s < n) pred[s] = t;
}
template <typename M>
__global__ void __launch_bounds__(CH_TB) ch_succ_vertex_kernel(M m, const u32 *__restrict__ pred, u32 n,
                                                                euler_succ_vertex *__restrict__ v)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    euler_succ_vertex x;
    x.vid = t;
    const u32 s = m.succ(t);
    x.n1 = s < n ? s : n;
    x.n2 = pred[t];
    v[t] = x;
}
static __global__ void __launch_bounds__(CH_TB) ch_fill_kernel(u32 *p, u64 n, u32 val)
{
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) p[t] = val;
}
static __global__ void __launch_bounds__(CH_TB) ch_has_start_kernel(const u32 *__restrict__ pred, const u32 *__restrict__ D, u32 n,
                                                                    u32 *__restrict__ has_start)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n && pred[t] >= n) has_start[D[t]] = 1u;
}
// anc[i] = (ancestor << 32) | distance; heads point to themselves with distance 0.
// head_kind: 0 not a head (or head of a suppressed component), 1 path head, 2 cycle head
template <typename M>
__global__ void __launch_bounds__(CH_TB) ch_rank_init_kernel(M m, const u32 *__restrict__ pred, const u32 *__restrict__ D,
                                                              const u32 *__restrict__ has_start, u32 n, u64 *__restrict__ anc,
                                                              u32 *__restrict__ head_kind)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u32 p = pred[t];
    u32 kind = 0;
    if (p >= n) kind = 1;
    else if (D[t] == t && !has_start[t]) kind = 2;
    anc[t] = kind ? ((u64)t << 32) : (((u64)p << 32) | 1ull);
    if (kind && !m.emit(D, t)) kind = 0;
    head_kind[t] = kind;
}
static __global__ void __launch_bounds__(CH_TB) ch_rank_step_kernel(const u64 *__restrict__ in, u64 *__restrict__ out, u32 n,
                                                                    u32 *changed)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u64 a = in[t];
    const u32 anc = (u32)(a >> 32);
    const u64 b = in[anc];
    const u32 anc2 = (u32)(b >> 32);
    if (anc2 != anc) {
        out[t] = ((u64)anc2 << 32) | (u64)((u32)a + (u32)b);
        *changed = 1u;
    } else {
        out[t] = a;  // ancestor already is the head
    }
}
struct ChKindIn {
    const u32 *k;
    u32 want;
    __device__ __forceinline__ u32 operator()(u64 i) const { return k[i] == want ? 1u : 0u; }
};
template <typename M>
__global__ void __launch_bounds__(CH_TB) ch_len_kernel(M m, const u32 *__restrict__ head_kind, const u64 *__restrict__ anc,
                                                        const u32 *__restrict__ ord1, const u32 *__restrict__ ord2, u32 n_starts,
                                                        u32 n, u32 k, u32 *__restrict__ len_by_ord)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u32 head = (u32)(anc[t] >> 32);
    const u32 hk = head_kind[head];
    if (!hk) return;
    const u32 s = m.succ(t);
    const bool tail = (s >= n) || (s == head);  // s == head only happens on a (cut) cycle
    if (!tail) return;
    const u32 dist = (u32)anc[t];
    const u32 ord = hk == 1 ? ord1[head] : n_starts + ord2[head];
    len_by_ord[ord] = k + dist + M::HEAD_APPENDS + 1;  // k-mer + appended bases + '\n'
}
template <typename M>
__global__ void __launch_bounds__(CH_TB) ch_write_kernel(M m, const u32 *__restrict__ head_kind, const u64 *__restrict__ anc,
                                                          const u32 *__restrict__ ord1, const u32 *__restrict__ ord2,
                                                          u32 n_starts, u32 n, u32 k, const u64 *__restrict__ off_by_ord,
                                                          const u32 *__restrict__ len_by_ord, char *__restrict__ out)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u32 head = (u32)(anc[t] >> 32), dist = (u32)anc[t];
    const u32 hk = head_kind[head];
    if (!hk) return;
    const u32 ord = hk == 1 ? ord1[head] : n_starts + ord2[head];
    const u64 o = off_by_ord[ord];
    if (M::HEAD_APPENDS || t != head) out[o + k + dist - (1 - M::HEAD_APPENDS)] = m.base(t);
    if (t == head) {
        u64 x = m.head_key(t), xh = m.head_key_hi(t);  // getString eulercuda.py:315-321
        for (u32 i = 0; i < k; i++) {
            out[o + k - 1 - i] = "ACGT"[x & 3];
            x = (x >> 2) | (xh << 62);
            xh >>= 2;
        }
        out[o + len_by_ord[ord] - 1] = '\n';
    }
}
// u32 lengths -> u64 offsets: two-level (tile sums are u32-safe because a tile is 4096 contigs)
struct ChLenIn {
    const u32 *p;
    __device__ __forceinline__ u32 operator()(u64 i) const { return p[i]; }
};
static __global__ void __launch_bounds__(CH_TB) ch_widen_kernel(const u32 *__restrict__ in, u64 n, u64 *__restrict__ out)
{
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = in[t];
}

// The ranking half of chain_emit, kept in one place for the callers that also need the ranks (clean.cu): predecessor
// scatter, components, head kinds and anc.  After chain_rank, anc is ancA or ancB.
struct ChainRanks {
    DevTmp<u32> pred, D, has_start, head_kind, ord1, ord2, changed;
    DevTmp<euler_succ_vertex> sv;
    DevTmp<u64> ancA, ancB, totals;
    u64 *anc = nullptr;
    ChainRanks(euler_ctx *ctx, u32 n)
        : pred(ctx, n), D(ctx, n), has_start(ctx, n), head_kind(ctx, n), ord1(ctx, n), ord2(ctx, n), changed(ctx, 1), sv(ctx, n),
          ancA(ctx, n), ancB(ctx, n), totals(ctx, 4)
    {
    }
    bool ok() const
    {
        return pred.ok() && D.ok() && has_start.ok() && head_kind.ok() && ord1.ok() && ord2.ok() && changed.ok() && sv.ok() &&
               ancA.ok() && ancB.ok() && totals.ok();
    }
};
#define CHAIN_RANKS_CHECK(ctx, r)                                                                   \
    do {                                                                                           \
        if (!(r).ok()) return euler_fail((ctx), EULER_ERR_NOMEM, "%s:%d device temp alloc failed", __FILE__, __LINE__); \
    } while (0)

template <typename M>
static int chain_rank(euler_ctx *ctx, M m, u32 n, ChainRanks &r)
{
    const unsigned g = grid_for(n, CH_TB);
    cudaStream_t s = ctx->stream;
    ch_fill_kernel<<<g, CH_TB, 0, s>>>(r.pred, n, n);
    ch_pred_kernel<<<g, CH_TB, 0, s>>>(m, n, r.pred);
    ch_succ_vertex_kernel<<<g, CH_TB, 0, s>>>(m, r.pred, n, r.sv);
    EULER_TRY(tour_components(ctx, r.sv, n, r.D));
    CUDA_TRY(ctx, cudaMemsetAsync(r.has_start, 0, (size_t)n * 4, s));
    ch_has_start_kernel<<<g, CH_TB, 0, s>>>(r.pred, r.D, n, r.has_start);
    ch_rank_init_kernel<<<g, CH_TB, 0, s>>>(m, r.pred, r.D, r.has_start, n, r.ancA, r.head_kind);
    CUDA_TRY(ctx, cudaGetLastError());
    u64 *cur = r.ancA, *nxt = r.ancB;
    for (int round = 0; round < 40; round++) {
        CUDA_TRY(ctx, cudaMemsetAsync(r.changed, 0, 4, s));
        ch_rank_step_kernel<<<g, CH_TB, 0, s>>>(cur, nxt, n, r.changed);
        CUDA_TRY(ctx, cudaMemcpyAsync(ctx->h_pinned, r.changed.get(), 4, cudaMemcpyDeviceToHost, s));
        CUDA_TRY(ctx, cudaStreamSynchronize(s));
        u64 *t = cur; cur = nxt; nxt = t;
        if (!*(u32 *)ctx->h_pinned) break;
    }
    r.anc = cur;
    return EULER_OK;
}

// The emitting half on ranks of the same model: contig order (ord1 / ord2, *n_starts = number of path contigs),
// lengths, text.  Emits into ctx->text_buf.  keep_off (may be NULL): the contig offsets on the device, with the text
// bytes as entry ncontigs.
template <typename M>
static int chain_spell(euler_ctx *ctx, M m, u32 n, u32 k, ChainRanks &r, char **d_out, u64 *out_bytes, u64 *ncontigs,
                       u32 *n_starts = nullptr, DevArr<u64> *keep_off = nullptr)
{
    const unsigned g = grid_for(n, CH_TB);
    cudaStream_t s = ctx->stream;
    u64 *cur = r.anc;
    EULER_TRY(scan_exclusive(ctx, ChKindIn{r.head_kind, 1u}, n, r.ord1.get(), r.totals.get() + 0));
    EULER_TRY(scan_exclusive(ctx, ChKindIn{r.head_kind, 2u}, n, r.ord2.get(), r.totals.get() + 1));
    u64 h[2];
    EULER_TRY(read_u64s(ctx, r.totals, h, 2));
    if (n_starts) *n_starts = (u32)h[0];
    const u64 nc = h[0] + h[1];
    if (!nc) return EULER_OK;
    DevTmp<u32> len_by_ord(ctx, nc), off32(ctx, nc);
    DevTmp<u64> off_by_ord(ctx, nc);
    TMP_CHECK(ctx, len_by_ord); TMP_CHECK(ctx, off32); TMP_CHECK(ctx, off_by_ord);
    ch_len_kernel<<<g, CH_TB, 0, s>>>(m, r.head_kind, cur, r.ord1, r.ord2, (u32)h[0], n, k, len_by_ord);
    EULER_TRY(scan_exclusive(ctx, ChLenIn{len_by_ord}, nc, off32.get(), r.totals.get() + 2));
    u64 bytes = 0;
    EULER_TRY(read_u64(ctx, r.totals.get() + 2, &bytes));
    if (bytes >= 0xffffffffull)
        return euler_fail(ctx, EULER_ERR_RANGE, "contig text of %llu bytes exceeds the 4 GiB emission limit", bytes);
    ch_widen_kernel<<<grid_for(nc, CH_TB), CH_TB, 0, s>>>(off32, nc, off_by_ord);
    EULER_TRY(dev_reserve(ctx, ctx->text_buf, bytes));
    ch_write_kernel<<<g, CH_TB, 0, s>>>(m, r.head_kind, cur, r.ord1, r.ord2, (u32)h[0], n, k, off_by_ord, len_by_ord,
                                        (char *)ctx->text_buf.p);
    CUDA_TRY(ctx, cudaGetLastError());
    if (keep_off) {
        EULER_TRY(keep_off->reserve(ctx, nc + 1));
        CUDA_TRY(ctx, cudaMemcpyAsync(keep_off->ptr(), off_by_ord.get(), nc * sizeof(u64), cudaMemcpyDeviceToDevice, s));
        CUDA_TRY(ctx, cudaMemcpyAsync(keep_off->ptr() + nc, r.totals.get() + 2, sizeof(u64), cudaMemcpyDeviceToDevice, s));
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    ctx->text_gen++;
    *d_out = (char *)ctx->text_buf.p;
    *out_bytes = bytes;
    *ncontigs = nc;
    return EULER_OK;
}

// Emits into ctx->text_buf.  Total text must stay below 4 GiB (u32 scan); larger jobs are split
// by the caller.
template <typename M>
static int chain_emit(euler_ctx *ctx, M m, u32 n, u32 k, char **d_out, u64 *out_bytes, u64 *ncontigs)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0;
    if (!n) return EULER_OK;
    ChainRanks r(ctx, n);
    CHAIN_RANKS_CHECK(ctx, r);
    EULER_TRY(chain_rank(ctx, m, n, r));
    return chain_spell(ctx, m, n, k, r, d_out, out_bytes, ncontigs);
}
