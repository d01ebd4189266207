// Top-k target retrieval over all nodes: the source sweep (every node as a candidate target of every query) expanded
// into a batch's links, and the fold of a batch's scores into per-query top-k state and filtered-rank counters.
#include <cooperative_groups.h>
#include <math.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace lpf {

constexpr int kTopkTile = 4096;      // scores per stage-A CTA (a tile never spans two queries)
constexpr int kTopkThreadsA = 512;
constexpr int kTopkThreadsB = 1024;
constexpr int kTopkMaxK = 1024;
constexpr int kExStage = 2048;       // exclusion-row ids staged in shared memory; a longer (hub) row is searched in global

// ---------------------------------------------------------------------------------------
// Source sweep -> link pairs: flat link i = q n_targets + j is (source[q], j).  Writes the flat range of n links that
// starts at position j0 of its first query: links[0, i] = source[(j0 + i) / n_targets], links[1, i] = (j0 + i) %
// n_targets.  A source outside [0, num_nodes) is written as 0 and raises *bad.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) expand_source_sweep_kernel(const T* __restrict__ source, int64_t nt, int64_t j0,
                                                                  int64_t n, int64_t num_nodes,
                                                                  int64_t* __restrict__ links, int64_t ld,
                                                                  int64_t* __restrict__ bad) {
    bool flag = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t p = j0 + i;
        const int64_t q = p / nt;
        const int64_t s = (int64_t)__ldg(source + q);
        const bool ok = s >= 0 && s < num_nodes;
        links[i] = ok ? s : 0;
        links[ld + i] = p - q * nt;
        flag |= !ok;
    }
    if (__any_sync(kFull, flag) && (threadIdx.x & 31) == 0) *bad = 1;
}

// ---------------------------------------------------------------------------------------
// Top-k fold.  A candidate (score s, target j) is the 64-bit key  ord(s) << 32 | ~j : unsigned order of the keys is
// (score descending, id ascending), keys of one query are unique, and 0 (an empty slot) is below every candidate.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ord_key(float f) {
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord_val(uint32_t o) { return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o); }
__device__ __forceinline__ uint64_t cand_key(float s, int64_t j) {
    return ((uint64_t)ord_key(s) << 32) | (uint32_t)~(uint32_t)j;
}
__device__ __forceinline__ uint64_t slot_key(const float* key, const int32_t* id, int i) {
    const int32_t j = id[i];
    return j >= 0 ? cand_key(key[i], j) : 0ull;
}

struct SelectSmem {
    unsigned hist[256];
    unsigned wsum[8];
    unsigned res[3];
};

// Radix select over the keys every thread hands to f(key) through visit(f) (blockDim >= 256): returns the smallest t
// >= 1 such that the non-zero keys >= t are exactly the min(k, #non-zero) largest.  Eight passes of 8 bits at most;
// a pass stops the search when the whole bucket holding the k-th key is taken.
template <typename Visit>
__device__ uint64_t block_select(Visit visit, int k, SelectSmem& sm) {
    uint64_t prefix = 0, mask = 0;
    unsigned need = (unsigned)k;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int i = tid; i < 256; i += blockDim.x) sm.hist[i] = 0;
        __syncthreads();
        visit([&](uint64_t key) {       // one atomic per bucket and warp: keys of one query often share their top bytes
            const bool hit = key != 0 && (key & mask) == prefix;
            const unsigned bin = hit ? (unsigned)((key >> shift) & 255) : 256u + (threadIdx.x & 31);
            const cg::coalesced_group same = cg::labeled_partition(cg::coalesced_threads(), bin);
            if (hit && same.thread_rank() == 0) atomicAdd(&sm.hist[bin], same.size());
        });
        __syncthreads();
        unsigned c = 0, incl = 0;
        if (tid < 256) {                       // thread t holds bucket 255 - t: inclusive sums from the top bucket down
            c = sm.hist[255 - tid];
            incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned y = __shfl_up_sync(kFull, incl, o);
                if (lane >= o) incl += y;
            }
            if (lane == 31) sm.wsum[warp] = incl;
        }
        __syncthreads();
        if (tid < 256) {
            for (int w = 0; w < warp; ++w) incl += sm.wsum[w];
            const unsigned excl = incl - c;
            if (excl < need && incl >= need) {
                sm.res[0] = 255 - tid;
                sm.res[1] = excl;
                sm.res[2] = c;
            }
            if (tid == 255 && incl < need) sm.res[0] = 256;      // (first pass only) fewer than k keys in all
        }
        __syncthreads();
        const unsigned b = sm.res[0], above = sm.res[1], cnt = sm.res[2];
        __syncthreads();                       // (res is rewritten by the next pass)
        if (b == 256) return 1;
        prefix |= (uint64_t)b << shift;
        mask |= (uint64_t)255 << shift;
        need -= above;
        if (cnt == need) return prefix;        // every key with this prefix is taken
    }
    return prefix;
}

__device__ __forceinline__ bool in_sorted(const int32_t* a, int64_t n, int32_t key, bool shared) {
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int32_t v = shared ? a[mid] : __ldg(a + mid);
        if (v < key) lo = mid + 1; else hi = mid;
    }
    return lo < n && (shared ? a[lo] : __ldg(a + lo)) == key;
}

// Stage A: one CTA per tile of <= kTopkTile scores of one query.  Counts the candidates against the positive's score
// (one 64-bit atomic per counter and CTA: the sums do not depend on the order), drops the keys below the query's
// stored k-th best (stale is fine: it only rises), selects the tile's top min(k, kept) and writes them to the tile's
// own kcap slots of the workspace (the rest zeroed: empty).  Exclusion is looked up only for scores that pass one of
// the two thresholds.
template <typename T>
__global__ void __launch_bounds__(kTopkThreadsA) topk_tiles_kernel(
    const float* __restrict__ prob, int64_t lo, int64_t n, const T* __restrict__ source, int64_t nt,
    const int64_t* __restrict__ ex_rowptr, const int32_t* __restrict__ ex_col, int64_t ex_rows,
    const T* __restrict__ positive, const float* __restrict__ pos_score, int k, const float* __restrict__ top_key,
    const int32_t* __restrict__ top_id, unsigned long long* __restrict__ cnt_ge, unsigned long long* __restrict__ cnt_gt,
    const int64_t* __restrict__ skip, int64_t tiles_per_query, int64_t g0, int kcap, uint64_t* __restrict__ ws_keys) {
    if (skip != nullptr && *skip != 0) return;
    __shared__ uint64_t keys[kTopkTile];
    __shared__ int32_t exrow[kExStage];
    __shared__ SelectSmem sm;
    __shared__ unsigned long long red[2];
    __shared__ int nlive, nsel;
    const int tid = threadIdx.x;
    const int64_t g = g0 + blockIdx.x;
    const int64_t q = g / tiles_per_query;
    const int64_t base = q * nt;
    int64_t jb = (g - q * tiles_per_query) * kTopkTile, je = min(jb + (int64_t)kTopkTile, nt);
    jb = max(jb, lo - base);
    je = min(je, lo + n - base);
    const int len = (int)(je - jb);
    const int64_t s = (int64_t)source[q];
    const int32_t* row = nullptr;
    int64_t rlen = 0;
    if (ex_rowptr != nullptr && s >= 0 && s < ex_rows) {
        const int64_t r0 = ex_rowptr[s];
        rlen = ex_rowptr[s + 1] - r0;
        row = ex_col + r0;
    }
    const bool staged = rlen <= kExStage;
    if (staged)
        for (int i = tid; i < rlen; i += blockDim.x) exrow[i] = row[i];
    if (tid == 0) {
        red[0] = red[1] = 0;
        nlive = nsel = 0;
    }
    const uint64_t thr = slot_key(top_key + q * k, top_id + q * k, k - 1);
    const bool has_pos = positive != nullptr;
    const float ps = has_pos ? pos_score[q] : 0.f;
    const int64_t pj = has_pos ? (int64_t)positive[q] : -1;
    __syncthreads();
    unsigned long long ge = 0, gt = 0;
    unsigned live = 0;
    for (int i = tid; i < len; i += blockDim.x) {
        const int64_t j = jb + i;
        const float sc = __ldg(prob + (base + j - lo));
        const uint64_t key = cand_key(sc, j);
        const bool counted = has_pos && sc >= ps && j != pj;
        const bool top = key > thr;
        bool ok = j != s;
        if (ok && (counted || top) && rlen > 0) ok = !in_sorted(staged ? exrow : row, rlen, (int32_t)j, staged);
        if (ok && counted) {
            ++ge;
            gt += sc > ps;
        }
        const uint64_t kk = (ok && top) ? key : 0ull;
        keys[i] = kk;
        live += kk != 0;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ge += __shfl_xor_sync(kFull, ge, o);
        gt += __shfl_xor_sync(kFull, gt, o);
        live += __shfl_xor_sync(kFull, live, o);
    }
    if ((tid & 31) == 0) {
        if (ge) atomicAdd(&red[0], ge);
        if (gt) atomicAdd(&red[1], gt);
        if (live) atomicAdd(&nlive, (int)live);
    }
    __syncthreads();
    if (tid == 0 && has_pos) {
        if (red[0]) atomicAdd(cnt_ge + q, red[0]);
        if (red[1]) atomicAdd(cnt_gt + q, red[1]);
    }
    const int m = nlive;
    uint64_t t = 1;
    if (m > k)
        t = block_select([&](auto f) { for (int i = tid; i < len; i += blockDim.x) f(keys[i]); }, k, sm);
    uint64_t* out = ws_keys + (int64_t)blockIdx.x * kcap;
    for (int i = tid; i < len; i += blockDim.x) {
        const uint64_t key = keys[i];
        if (key >= t) {
            const int p = atomicAdd(&nsel, 1);
            if (p < kcap) out[p] = key;
        }
    }
    __syncthreads();
    for (int i = nsel + tid; i < kcap; i += blockDim.x) out[i] = 0;
}

// Stage B: one CTA per query the batch touches.  The top k of the stored state and of the survivors of the query's
// tiles, sorted by (score descending, id ascending) and written back; unfilled slots stay (-inf, -1).
__global__ void __launch_bounds__(kTopkThreadsB) topk_merge_kernel(int64_t q0, int64_t tiles_per_query, int64_t g0,
                                                                   int64_t ntiles, int k, int kcap, float* top_key,
                                                                   int32_t* top_id, const uint64_t* __restrict__ ws_keys,
                                                                   const int64_t* __restrict__ skip) {
    if (skip != nullptr && *skip != 0) return;
    __shared__ uint64_t sel[kTopkMaxK];
    __shared__ SelectSmem sm;
    __shared__ int nsel;
    const int tid = threadIdx.x;
    const int64_t q = q0 + blockIdx.x;
    const int64_t a = max(q * tiles_per_query, g0) - g0, b = min((q + 1) * tiles_per_query, g0 + ntiles) - g0;
    float* tk = top_key + q * k;
    int32_t* ti = top_id + q * k;
    const uint64_t* slots = ws_keys + a * kcap;                 // the query's tiles' slots: one contiguous range
    const int64_t span = (b - a) * kcap;
    auto visit = [&](auto f) {
        for (int i = tid; i < k; i += blockDim.x) f(slot_key(tk, ti, i));
        for (int64_t i0 = tid; i0 < span; i0 += 4 * (int64_t)blockDim.x) {
            uint64_t v[4];                                      // four loads in flight per thread
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t i = i0 + (int64_t)u * blockDim.x;
                v[u] = i < span ? __ldg(slots + i) : 0ull;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) f(v[u]);
        }
    };
    if (tid == 0) nsel = 0;
    const uint64_t t = block_select(visit, k, sm);          // (its barriers order nsel = 0 before the gather)
    visit([&](uint64_t key) {
        if (key >= t) {
            const int p = atomicAdd(&nsel, 1);
            if (p < k) sel[p] = key;
        }
    });
    __syncthreads();
    const int cnt = min(nsel, k);
    int P = 1;
    while (P < k) P <<= 1;
    for (int i = cnt + tid; i < P; i += blockDim.x) sel[i] = 0;
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {             // bitonic sort, descending
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = tid; i < P; i += blockDim.x) {
                const int l = i ^ stride;
                if (l > i) {
                    const uint64_t x = sel[i], y = sel[l];
                    if (((i & size) == 0) ? (x < y) : (x > y)) {
                        sel[i] = y;
                        sel[l] = x;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int i = tid; i < k; i += blockDim.x) {
        const uint64_t key = sel[i];
        tk[i] = key ? ord_val((uint32_t)(key >> 32)) : -INFINITY;
        ti[i] = key ? (int32_t)~(uint32_t)key : -1;
    }
}

}  // namespace lpf

using namespace lpf;

extern "C" int lpf_expand_source_sweep(const void* source, int32_t id_bytes, int64_t n_targets, int64_t j0, int64_t n,
                                       int64_t num_nodes, int64_t* links, int64_t ld, int64_t* bad, void* stream) {
    LPF_REQUIRE(id_bytes == 4 || id_bytes == 8, "id_bytes must be 4 or 8");
    LPF_REQUIRE(n_targets >= 1, "n_targets must be >= 1");
    LPF_REQUIRE(n >= 0 && j0 >= 0 && j0 < n_targets, "bad range (need n >= 0, 0 <= j0 < n_targets)");
    LPF_REQUIRE(num_nodes >= n_targets, "n_targets > num_nodes (targets must be node ids)");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(source && links && bad, "NULL argument");
    LPF_REQUIRE(ld >= n, "ld < n");
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)kNumSMs * 8;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    if (id_bytes == 4)
        expand_source_sweep_kernel<int32_t><<<(unsigned)blocks, 256, 0, st>>>((const int32_t*)source, n_targets, j0, n,
                                                                             num_nodes, links, ld, bad);
    else
        expand_source_sweep_kernel<int64_t><<<(unsigned)blocks, 256, 0, st>>>((const int64_t*)source, n_targets, j0, n,
                                                                             num_nodes, links, ld, bad);
    return check_launch("lpf_expand_source_sweep");
}

static int64_t topk_tiles_max(int64_t n, int64_t n_targets) {
    // a range of n positions touches 1 tile plus one per tile or query boundary inside it
    return 1 + (n + kTopkTile - 1) / kTopkTile + (n + n_targets - 1) / n_targets;
}

extern "C" int64_t lpf_topk_fold_workspace_bytes(int64_t bs, int32_t k, int64_t n_targets) {
    if (bs < 0 || k < 1 || k > kTopkMaxK || n_targets < 1) return -1;
    const int64_t tiles = topk_tiles_max(bs, n_targets);
    const int64_t kcap = k < kTopkTile ? k : kTopkTile;
    return tiles * kcap * 8;
}

extern "C" int lpf_topk_fold(const float* prob, int64_t lo, int64_t n, const void* source, const void* positive,
                             int32_t id_bytes, int64_t num_queries, int64_t n_targets, const int64_t* ex_rowptr,
                             const int32_t* ex_col, int64_t ex_rows, const float* pos_score, int32_t k, float* top_key,
                             int32_t* top_id, int64_t* cnt_ge, int64_t* cnt_gt, const int64_t* skip, void* workspace,
                             int64_t workspace_bytes, void* stream) {
    LPF_REQUIRE(id_bytes == 4 || id_bytes == 8, "id_bytes must be 4 or 8");
    LPF_REQUIRE(k >= 1 && k <= kTopkMaxK, "k must be in [1, 1024]");
    LPF_REQUIRE(n_targets >= 1 && n_targets <= INT32_MAX, "n_targets must be in [1, 2^31)");
    LPF_REQUIRE(num_queries >= 0 && lo >= 0 && n >= 0, "bad range (need lo >= 0, n >= 0)");
    LPF_REQUIRE(lo + n <= num_queries * n_targets, "range past the last query");
    LPF_REQUIRE(ex_rows >= 0 && (ex_rowptr == nullptr) == (ex_col == nullptr),
                "exclusion: rowptr and col are given together");
    const bool has_pos = positive != nullptr;
    LPF_REQUIRE((pos_score != nullptr) == has_pos && (cnt_ge != nullptr) == has_pos && (cnt_gt != nullptr) == has_pos,
                "positive, pos_score, cnt_ge and cnt_gt are given together");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(prob && source && top_key && top_id && workspace, "NULL argument");
    LPF_REQUIRE(workspace_bytes >= lpf_topk_fold_workspace_bytes(n, k, n_targets),
                "workspace smaller than lpf_topk_fold_workspace_bytes(n, k, n_targets)");
    const int64_t tq = (n_targets + kTopkTile - 1) / kTopkTile;
    const int64_t last = lo + n - 1;
    const int64_t q0 = lo / n_targets, q1 = last / n_targets;
    const int64_t g0 = q0 * tq + (lo - q0 * n_targets) / kTopkTile;
    const int64_t g1 = q1 * tq + (last - q1 * n_targets) / kTopkTile;
    const int64_t ntiles = g1 - g0 + 1;
    const int kcap = k < kTopkTile ? k : kTopkTile;
    uint64_t* ws_keys = (uint64_t*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long *ge = (unsigned long long*)cnt_ge, *gt = (unsigned long long*)cnt_gt;
    if (id_bytes == 4)
        topk_tiles_kernel<int32_t><<<(unsigned)ntiles, kTopkThreadsA, 0, st>>>(
            prob, lo, n, (const int32_t*)source, n_targets, ex_rowptr, ex_col, ex_rows, (const int32_t*)positive,
            pos_score, k, top_key, top_id, ge, gt, skip, tq, g0, kcap, ws_keys);
    else
        topk_tiles_kernel<int64_t><<<(unsigned)ntiles, kTopkThreadsA, 0, st>>>(
            prob, lo, n, (const int64_t*)source, n_targets, ex_rowptr, ex_col, ex_rows, (const int64_t*)positive,
            pos_score, k, top_key, top_id, ge, gt, skip, tq, g0, kcap, ws_keys);
    int rc = check_launch("lpf_topk_fold (tiles)");
    if (rc != LPF_OK) return rc;
    topk_merge_kernel<<<(unsigned)(q1 - q0 + 1), kTopkThreadsB, 0, st>>>(q0, tq, g0, ntiles, k, kcap, top_key, top_id,
                                                                         ws_keys, skip);
    return check_launch("lpf_topk_fold (merge)");
}
