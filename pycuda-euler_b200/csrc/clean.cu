// clean.cu -- the link rule of unitig mode, and tip clipping, isolated-fragment removal and bubble popping on the
// unitig node graph, then emission.  With zero rounds it spells the plain unitigs.
//
// Key-independent: unitig.cu describes the node graph once, for either key width, as
//   nbr[4 i + b]  node id of the forward extension of node i by base b, or EULER_NO_ID (absent or filtered),
//   twin_id[i]    node id of the reverse complement,
//   cnt[i]        both-strand count (read only by the rounds and the sums),
// and the keys as 64-bit words (key_stride words per node, low word first) for spelling.  From then on everything
// is node ids.  Every round works on one snapshot of the alive mask:
//   1. succ: the link rule on alive nodes (the backward degree of y is the alive forward degree of twin(y); the
//      hairpin stop is cand == twin(x));
//   2. chain_rank (chain.cuh): every node knows its chain head and its distance to it;
//   3. per path unitig (indexed by its head): sum of counts, tail, L, cov, bubble end point;
//   4. decisions (rules in euler_b200.h), taken per head on the snapshot;
//   5. the removal scatter, on every node of a removed unitig and on its twin.
// Rules compare coverages strictly and sets by membership, so the outcome depends on the counts alone.
#include "chain.cuh"
#include "kernels.h"
#include "tmp.cuh"

#define CB 256

// node graph of one round, for chain.cuh.  emit: only alive nodes are written (a dead node is a single-node chain
// of its own), and each unitig once, on the strand whose component label is the smaller one.
struct CleanChainModel {
    const u64 *words;
    u32 stride;
    const u32 *succ_;
    const u32 *twin_id;
    const unsigned char *alive;
    static constexpr u32 HEAD_APPENDS = 0;
    __device__ __forceinline__ u32 succ(u32 i) const { return succ_[i]; }
    __device__ __forceinline__ u64 head_key(u32 i) const { return words[(u64)stride * i]; }
    __device__ __forceinline__ u64 head_key_hi(u32 i) const { return stride > 1 ? words[(u64)stride * i + 1] : 0ull; }
    __device__ __forceinline__ char base(u32 i) const { return "ACGT"[words[(u64)stride * i] & 3]; }
    __device__ __forceinline__ bool emit(const u32 *D, u32 i) const { return alive[i] && D[i] <= D[twin_id[i]]; }
};

// alive forward extensions of x: their number, the last one in *one
__device__ __forceinline__ u32 alive_fw(const u32 *nbr, const unsigned char *alive, u32 x, u32 *one)
{
    u32 d = 0;
    for (u32 b = 0; b < 4; b++) {
        const u32 y = nbr[4ull * x + b];
        if (y != EULER_NO_ID && alive[y]) { d++; *one = y; }
    }
    return d;
}

// referenceAssembler.get_contig_forward :59-77, one step, for every alive node: x -> y iff y is the only alive forward
// extension of x, x the only alive backward extension of y, and y is not twin(x) (hairpin stop, :70-71)
__global__ void __launch_bounds__(CB) clean_succ_kernel(const u32 *__restrict__ nbr, const u32 *__restrict__ twin_id,
                                                        const unsigned char *__restrict__ alive, u32 n, u32 *__restrict__ succ)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 s = n, cand = EULER_NO_ID, back = EULER_NO_ID;
    if (alive[i] && alive_fw(nbr, alive, i, &cand) == 1 && cand != twin_id[i] &&
        alive_fw(nbr, alive, twin_id[cand], &back) == 1)
        s = cand;
    succ[i] = s;
}

// node t of a path unitig: add its count to the unitig's sum, and record the tail.  Dead nodes and cycles are skipped.
__global__ void __launch_bounds__(CB) clean_sum_kernel(const u32 *__restrict__ succ, const u32 *__restrict__ pred,
                                                       const u64 *__restrict__ anc, const u32 *__restrict__ cnt,
                                                       const unsigned char *__restrict__ alive, u32 n, u64 *__restrict__ usum,
                                                       u32 *__restrict__ utail)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || !alive[t]) return;
    const u32 h = (u32)(anc[t] >> 32);
    if (pred[h] < n) return;   // the head of a cut cycle has a predecessor
    atomicAdd(usum + h, (u64)cnt[t]);
    if (succ[t] >= n) utail[h] = t;
}

__device__ __forceinline__ bool is_path_head(const u32 *pred, const unsigned char *alive, u32 n, u32 h)
{
    return alive[h] && pred[h] >= n;
}

// per path head h: cov (in place of the sum) and, for a bubble candidate (in = {P}, out = {S}, L <= bubble_len), S
__global__ void __launch_bounds__(CB) clean_cov_kernel(const u32 *__restrict__ nbr, const u32 *__restrict__ twin_id,
                                                       const unsigned char *__restrict__ alive, const u32 *__restrict__ pred,
                                                       const u64 *__restrict__ anc, const u32 *__restrict__ utail, u32 n,
                                                       u32 bubble_len, u64 *__restrict__ ucov, u32 *__restrict__ uS)
{
    const u32 h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n) return;
    u32 S = EULER_NO_ID;
    if (is_path_head(pred, alive, n, h)) {
        const u32 t = utail[h];
        const u32 L = (u32)anc[t] + 1u;
        // floor(65536 sum / L) without a 128-bit product: sum = q L + rem, rem < L < 2^32
        const u64 sum = ucov[h], q = sum / L, rem = sum - q * L;
        ucov[h] = (q << 16) + (rem << 16) / L;
        u32 z, s;
        if (L <= bubble_len && alive_fw(nbr, alive, twin_id[h], &z) == 1 && alive_fw(nbr, alive, t, &s) == 1) S = s;
    }
    uS[h] = S;
}

// largest cov of the unitigs headed by p's alive successors other than h; with S != EULER_NO_ID only those that are
// bubble candidates ending in S.  *any = whether there was one.
__device__ __forceinline__ u64 rival_cov(const u32 *nbr, const unsigned char *alive, const u64 *ucov, const u32 *uS, u32 p, u32 h,
                                         u32 S, bool *any)
{
    u64 m = 0;
    *any = false;
    for (u32 b = 0; b < 4; b++) {
        const u32 r = nbr[4ull * p + b];
        if (r == EULER_NO_ID || r == h || !alive[r]) continue;
        if (S != EULER_NO_ID && uS[r] != S) continue;
        *any = true;
        m = ucov[r] > m ? ucov[r] : m;
    }
    return m;
}

// stats: [0] tips, [1] isolated, [2] bubble branches (once per strand pair), [3] canonical K-mers removed
__global__ void __launch_bounds__(CB) clean_decide_kernel(const u32 *__restrict__ nbr, const u32 *__restrict__ twin_id,
                                                          const unsigned char *__restrict__ alive, const u32 *__restrict__ pred,
                                                          const u64 *__restrict__ anc, const u32 *__restrict__ utail,
                                                          const u64 *__restrict__ ucov, const u32 *__restrict__ uS, u32 n,
                                                          euler_clean_params p, unsigned char *__restrict__ rm,
                                                          u64 *__restrict__ stats)
{
    const u32 h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= n) return;
    u32 kind = 0;   // 1 tip, 2 isolated, 3 bubble branch
    if (is_path_head(pred, alive, n, h)) {
        const u32 t = utail[h];
        const u32 L = (u32)anc[t] + 1u;
        const u64 cov = ucov[h];
        u32 z = EULER_NO_ID, s = EULER_NO_ID;
        const u32 din = alive_fw(nbr, alive, twin_id[h], &z), dout = alive_fw(nbr, alive, t, &s);
        bool any = false;
        if (din == 0 && dout == 0) {
            if (L <= p.isolated_len) kind = 2;
        } else if (din == 1 && dout == 0) {
            if (L <= p.tip_len) {
                const u64 m = rival_cov(nbr, alive, ucov, uS, twin_id[z], h, EULER_NO_ID, &any);
                if (any && cov < m) kind = 1;
            }
        } else if (uS[h] != EULER_NO_ID) {
            const u64 m = rival_cov(nbr, alive, ucov, uS, twin_id[z], h, uS[h], &any);
            if (any && cov < m) kind = 3;
        }
        // a tip's twin is never removed by a rule of its own; isolated unitigs and bubble branches are removed on
        // both strands: count the strand whose head id is not larger than its twin's
        if (kind == 1 || (kind && h <= twin_id[t])) atomicAdd(stats + (kind - 1), 1ull);
    }
    rm[h] = (unsigned char)(kind != 0);
}

// every node of a removed unitig leaves the alive set with its twin; a canonical K-mer is counted by one thread
__global__ void __launch_bounds__(CB) clean_scatter_kernel(const u32 *__restrict__ twin_id, const u64 *__restrict__ anc,
                                                           const unsigned char *__restrict__ rm, u32 n,
                                                           unsigned char *__restrict__ alive, u64 *__restrict__ stats)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n || !rm[anc[t] >> 32]) return;
    const u32 tw = twin_id[t];
    alive[t] = 0;
    alive[tw] = 0;
    if (t <= tw || !rm[anc[tw] >> 32]) atomicAdd(stats + 3, 1ull);
}

// per emitted contig (output order of chain_spell): sum of its nodes' counts
__global__ void __launch_bounds__(CB) clean_contig_sums_kernel(const u64 *__restrict__ anc, const u32 *__restrict__ head_kind,
                                                               const u32 *__restrict__ ord1, const u32 *__restrict__ ord2,
                                                               u32 n_starts, const u32 *__restrict__ cnt, u32 n,
                                                               u64 *__restrict__ sums)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const u32 h = (u32)(anc[t] >> 32);
    const u32 hk = head_kind[h];
    if (!hk) return;
    atomicAdd(sums + (hk == 1 ? ord1[h] : n_starts + ord2[h]), (u64)cnt[t]);
}

static __global__ void __launch_bounds__(CB) clean_fill_kernel(unsigned char *p, u32 n, unsigned char v)
{
    const u32 t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) p[t] = v;
}

int clean_unitigs(euler_ctx *ctx, u32 n, u32 K, const u64 *key_words, u32 key_stride, const u32 *nbr, const u32 *twin_id,
                  const u32 *cnt, const euler_clean_params &p, char **d_out, u64 *out_bytes, u64 *ncontigs, u64 *h_sums,
                  u64 sums_cap, euler_clean_stats *st, UnitigsKept *keep)
{
    *d_out = nullptr; *out_bytes = 0; *ncontigs = 0;
    if (keep) keep->n_starts = 0;
    *st = euler_clean_stats{};
    if (!n) return EULER_OK;
    const u32 nr = p.max_rounds ? n : 0;   // rm, utail, uS and ucov serve the rounds only
    DevTmp<unsigned char> alive(ctx, n), rm(ctx, nr);
    DevTmp<u32> succ(ctx, n), utail(ctx, nr), uS(ctx, nr);
    DevTmp<u64> ucov(ctx, nr), stats(ctx, 4);
    TMP_CHECK(ctx, alive); TMP_CHECK(ctx, rm); TMP_CHECK(ctx, succ); TMP_CHECK(ctx, utail); TMP_CHECK(ctx, uS);
    TMP_CHECK(ctx, ucov); TMP_CHECK(ctx, stats);
    ChainRanks r(ctx, n);
    CHAIN_RANKS_CHECK(ctx, r);
    const unsigned g = grid_for(n, CB);
    cudaStream_t s = ctx->stream;
    clean_fill_kernel<<<g, CB, 0, s>>>(alive, n, 1);
    CUDA_TRY(ctx, cudaMemsetAsync(stats, 0, 4 * sizeof(u64), s));
    const CleanChainModel m = {key_words, key_stride, succ, twin_id, alive};
    bool ranked = false;   // succ and r describe the current alive set
    u64 removed = 0;
    for (u32 round = 0; round < p.max_rounds; round++) {
        clean_succ_kernel<<<g, CB, 0, s>>>(nbr, twin_id, alive, n, succ);
        CUDA_TRY(ctx, cudaGetLastError());
        EULER_TRY(chain_rank(ctx, m, n, r));
        ranked = true;
        CUDA_TRY(ctx, cudaMemsetAsync(ucov, 0, (size_t)n * sizeof(u64), s));
        clean_sum_kernel<<<g, CB, 0, s>>>(succ, r.pred, r.anc, cnt, alive, n, ucov, utail);
        clean_cov_kernel<<<g, CB, 0, s>>>(nbr, twin_id, alive, r.pred, r.anc, utail, n, p.bubble_len, ucov, uS);
        clean_decide_kernel<<<g, CB, 0, s>>>(nbr, twin_id, alive, r.pred, r.anc, utail, ucov, uS, n, p, rm, stats);
        clean_scatter_kernel<<<g, CB, 0, s>>>(twin_id, r.anc, rm, n, alive, stats);
        CUDA_TRY(ctx, cudaGetLastError());
        u64 h[4];
        EULER_TRY(read_u64s(ctx, stats, h, 4));
        st->tips = h[0]; st->isolated = h[1]; st->bubble_branches = h[2]; st->kmers_removed = h[3];
        if (h[3] == removed) break;
        removed = h[3];
        st->rounds++;
        ranked = false;
    }
    if (!ranked) {
        clean_succ_kernel<<<g, CB, 0, s>>>(nbr, twin_id, alive, n, succ);
        CUDA_TRY(ctx, cudaGetLastError());
        EULER_TRY(chain_rank(ctx, m, n, r));
    }
    u32 n_starts = 0;
    EULER_TRY(chain_spell(ctx, m, n, K, r, d_out, out_bytes, ncontigs, &n_starts, keep ? &keep->off : nullptr));
    if (keep) keep->n_starts = n_starts;
    if ((!h_sums && !keep) || !*ncontigs) return EULER_OK;
    if (h_sums && sums_cap < *ncontigs)
        return euler_fail(ctx, EULER_ERR_ARG, "kmer_sums capacity too small (%llu < %llu)", sums_cap, *ncontigs);
    DevTmp<u64> tmp_sums(ctx, keep ? 0 : *ncontigs);
    TMP_CHECK(ctx, tmp_sums);
    if (keep) EULER_TRY(keep->sums.reserve(ctx, *ncontigs));
    u64 *sums = keep ? keep->sums.ptr() : tmp_sums.get();
    CUDA_TRY(ctx, cudaMemsetAsync(sums, 0, *ncontigs * sizeof(u64), s));
    clean_contig_sums_kernel<<<g, CB, 0, s>>>(r.anc, r.head_kind, r.ord1, r.ord2, n_starts, cnt, n, sums);
    CUDA_TRY(ctx, cudaGetLastError());
    if (h_sums) CUDA_TRY(ctx, cudaMemcpyAsync(h_sums, sums, *ncontigs * sizeof(u64), cudaMemcpyDeviceToHost, s));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return EULER_OK;
}
