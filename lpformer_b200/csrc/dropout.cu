// Dropout of the training path (rule and sites: include/lpformer_b200.h, "Dropout"; random numbers: common.cuh).
//   lpf_dropout            Y = X * mask / (1 - p) over strided rows: the forward of the feature, attention-output,
//                          score-head and MLP sites, the backward of every site (the same mask on dY), and the
//                          inspection hook (applied to ones it returns mask / (1 - p)).  Masks are never stored.
//   lpf_drop_pairs_count   node dropout (reference compute_node_mask -> drop_pairwise): a radix select of the K-th
//   lpf_drop_pairs_fill    smallest 64-bit pair key, the per-(type, link) counts of the kept pairs, then a stable
//                          compaction that keeps the type-major, (link, node)-sorted order.
#include "common.cuh"

namespace lpf {

__global__ void __launch_bounds__(256) dropout_kernel(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t rows,
                                                      int n, int64_t row0, const uint64_t* __restrict__ seed_p, int site,
                                                      uint64_t thr, float scale) {
    const uint64_t seed = *seed_p;
    const int groups = (n + 3) >> 2;
    const int64_t total = rows * groups;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / groups;
        const int g = (int)(e - r * groups);
        const uint4 u = dropout_bits(seed, site, row0 + r, g);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int c = 4 * g + j;
            if (c < n) Y[r * ldy + c] = dropout_apply(X[r * ldx + c], uint4_word(u, j), thr, scale);
        }
    }
}

// ------------------------------------------------------------------------------------------------------ node dropout
// Pair i of the selection gets the key (64 Philox bits of (seed, site, row i, col 0) with the low `bits` bits replaced
// by i), so keys are distinct and ties of the random part are broken by pair index; the K pairs of smallest key are a
// uniform K-subset.  Workspace: hist[256] (uint32), then state = (key prefix found so far, rank left within it).
struct DropState {
    uint32_t hist[256];
    uint64_t prefix;
    uint64_t rank;
    uint64_t none;       // K = 0: nothing is kept
};

__device__ __forceinline__ uint64_t pair_key(uint64_t seed, int site, int64_t i, int bits) {
    const uint4 u = dropout_bits(seed, site, i, 0);
    const uint64_t low = (1ull << bits) - 1;
    return ((((uint64_t)u.x << 32) | u.y) & ~low) | (uint64_t)i;
}

__global__ void drop_init_kernel(DropState* st, int64_t K) {
    st->hist[threadIdx.x] = 0;
    if (threadIdx.x == 0) {
        st->prefix = 0;
        st->rank = (uint64_t)K;          // 1-based rank of the K-th smallest key
        st->none = K == 0;
    }
}

// histogram of key bits [shift, shift + 8) over the keys whose bits above shift + 8 equal the prefix
__global__ void __launch_bounds__(256) drop_hist_kernel(int64_t S, const uint64_t* __restrict__ seed_p, int site, int bits,
                                                        int shift, DropState* st) {
    __shared__ uint32_t h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const uint64_t seed = *seed_p;
    const uint64_t hi = shift >= 56 ? 0ull : (~0ull << (shift + 8));
    const uint64_t prefix = st->prefix;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < S; i += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = pair_key(seed, site, i, bits);
        if ((k & hi) == prefix) atomicAdd(&h[(k >> shift) & 255], 1u);
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], h[threadIdx.x]);
}

// the bin holding the rank-th key: fixes 8 more bits of the prefix; clears the histogram for the next pass
__global__ void drop_pick_kernel(DropState* st, int shift) {
    if (threadIdx.x == 0) {
        uint64_t rank = st->rank, below = 0;
        int b = 0;
        for (; b < 255; ++b) {
            if (below + st->hist[b] >= rank) break;
            below += st->hist[b];
        }
        st->rank = rank - below;
        st->prefix |= (uint64_t)b << shift;
    }
    __syncthreads();
    st->hist[threadIdx.x] = 0;
}

// one warp per (type, link) segment: kept pairs (key <= the K-th smallest)
__global__ void __launch_bounds__(256) drop_count_kernel(const int64_t* __restrict__ ptr, int64_t segs,
                                                         const uint64_t* __restrict__ seed_p, int site, int bits,
                                                         const DropState* __restrict__ st, int32_t* __restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t seed = *seed_p, T = st->prefix;
    const bool none = st->none;
    for (int64_t s = warp; s < segs; s += nwarps) {
        const int64_t k0 = ptr[s], k1 = ptr[s + 1];
        int c = 0;
        for (int64_t i = k0 + lane; i < k1 && !none; i += 32) c += pair_key(seed, site, i, bits) <= T;
        c = __reduce_add_sync(kFull, c);
        if (lane == 0) counts[s] = c;
    }
}

__global__ void __launch_bounds__(256) drop_fill_kernel(const int64_t* __restrict__ ptr, int64_t segs,
                                                        const uint64_t* __restrict__ seed_p, int site, int bits,
                                                        const DropState* __restrict__ st,
                                                        const int32_t* __restrict__ node, const float* __restrict__ pa,
                                                        const float* __restrict__ pb, const int32_t* __restrict__ link,
                                                        const int64_t* __restrict__ ptr_out, int32_t* __restrict__ node_out,
                                                        float* __restrict__ pa_out, float* __restrict__ pb_out,
                                                        int32_t* __restrict__ link_out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const uint64_t seed = *seed_p, T = st->prefix;
    const unsigned below = (1u << lane) - 1u;
    if (st->none) return;
    for (int64_t s = warp; s < segs; s += nwarps) {
        const int64_t k1 = ptr[s + 1];
        int64_t o = ptr_out[s];
        for (int64_t i0 = ptr[s]; i0 < k1; i0 += 32) {
            const int64_t i = i0 + lane;
            const bool keep = i < k1 && pair_key(seed, site, i, bits) <= T;
            const unsigned m = __ballot_sync(kFull, keep);
            if (keep) {
                const int64_t j = o + __popc(m & below);
                node_out[j] = node[i];
                pa_out[j] = pa[i];
                pb_out[j] = pb[i];
                if (link) link_out[j] = link[i];
            }
            o += __popc(m);
        }
    }
}

static int key_bits(int64_t S) {
    int b = 1;
    while (b < 62 && (1ll << b) < S) ++b;
    return b;
}

static unsigned grid_for(int64_t items, int per_block, int64_t cap) {
    int64_t blocks = (items + per_block - 1) / per_block;
    if (blocks > cap) blocks = cap;
    return (unsigned)(blocks < 1 ? 1 : blocks);
}

}  // namespace lpf

using namespace lpf;

extern "C" int lpf_dropout(const float* X, int64_t ldx, float* Y, int64_t ldy, int64_t rows, int32_t n, int64_t row0,
                           const uint64_t* seed, int32_t site, double p, void* stream) {
    uint64_t thr;
    float scale;
    LPF_REQUIRE(dropout_rule(p, &thr, &scale), "p must be in [0, 1]");
    LPF_REQUIRE(rows >= 0 && n >= 1 && row0 >= 0, "bad shape");
    LPF_REQUIRE(seed, "seed is NULL");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(X && Y, "NULL argument");
    LPF_REQUIRE(ldx >= n && ldy >= n, "leading dimension too small");
    const int64_t groups = rows * ((n + 3) / 4);
    dropout_kernel<<<grid_for(groups, 256, (int64_t)kNumSMs * 16), 256, 0, (cudaStream_t)stream>>>(
        X, ldx, Y, ldy, rows, n, row0, seed, site, thr, scale);
    return check_launch("lpf_dropout");
}

extern "C" int64_t lpf_drop_pairs_workspace_bytes(void) { return (int64_t)sizeof(DropState); }

extern "C" int lpf_drop_pairs_count(const int64_t* ptr, int64_t bs, int64_t S, int64_t K, const uint64_t* seed,
                                    int32_t site, int32_t* counts, void* workspace, int64_t workspace_bytes,
                                    void* stream) {
    LPF_REQUIRE(bs >= 0 && S >= 0 && K >= 0 && K <= S, "bad sizes (need 0 <= K <= S)");
    LPF_REQUIRE(S < (1ll << 40), "S must be below 2^40");
    LPF_REQUIRE(workspace && workspace_bytes >= (int64_t)sizeof(DropState), "workspace too small");
    if (bs == 0) return LPF_OK;
    LPF_REQUIRE(ptr && counts && seed, "NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    DropState* ds = (DropState*)workspace;
    const int bits = key_bits(S);
    drop_init_kernel<<<1, 256, 0, st>>>(ds, K);
    if (K > 0) {
        const unsigned grid = grid_for(S, 256, (int64_t)kNumSMs * 8);
        for (int shift = 56; shift >= 0; shift -= 8) {
            drop_hist_kernel<<<grid, 256, 0, st>>>(S, seed, site, bits, shift, ds);
            drop_pick_kernel<<<1, 256, 0, st>>>(ds, shift);
        }
    }
    drop_count_kernel<<<grid_for(3 * bs, 8, (int64_t)kNumSMs * 16), 256, 0, st>>>(ptr, 3 * bs, seed, site, bits, ds, counts);
    return check_launch("lpf_drop_pairs_count");
}

extern "C" int lpf_drop_pairs_fill(const int64_t* ptr, int64_t bs, const int32_t* node, const float* src_ppr,
                                   const float* tgt_ppr, const int32_t* link, int64_t S, const uint64_t* seed,
                                   int32_t site, const void* workspace, const int64_t* ptr_out, int32_t* node_out,
                                   float* src_out, float* tgt_out, int32_t* link_out, void* stream) {
    LPF_REQUIRE(bs >= 0 && S >= 0, "bad sizes");
    LPF_REQUIRE(S < (1ll << 40), "S must be below 2^40");
    if (bs == 0 || S == 0) return LPF_OK;
    LPF_REQUIRE(ptr && node && src_ppr && tgt_ppr && seed && workspace && ptr_out && node_out && src_out && tgt_out,
                "NULL argument");
    LPF_REQUIRE((link == nullptr) == (link_out == nullptr), "link and link_out must both be given or both NULL");
    drop_fill_kernel<<<grid_for(3 * bs, 8, (int64_t)kNumSMs * 16), 256, 0, (cudaStream_t)stream>>>(
        ptr, 3 * bs, seed, site, key_bits(S), (const DropState*)workspace, node, src_ppr, tgt_ppr, link, ptr_out, node_out,
        src_out, tgt_out, link_out);
    return check_launch("lpf_drop_pairs_fill");
}
