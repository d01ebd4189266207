// Dense pieces of the path: RPE hidden vectors, the fp32 contraction, row-wise
// LayerNorm(+ReLU,+residual) and the link-level gathers.
#include "common.cuh"

namespace lpf {

// ---------------------------------------------------------------------------------------
// RPE hidden:  hsum[s,:] = h(pa,pb) + h(pb,pa),  h(x,y) = ReLU(LN_d(W1 [x,y]^T + b1))
// (get_pos_encodings, reference models/link_transformer.py:182-211, with the MLP of
// models/other_models.py:125-133).  One warp per pair, channels strided over lanes, the
// five per-channel parameters live in registers for the whole grid-stride loop.
// ---------------------------------------------------------------------------------------
template <int KC>
__global__ void __launch_bounds__(256) rpe_hidden_kernel(const float* __restrict__ pa, const float* __restrict__ pb,
                                                         int64_t row0, int64_t rows, const float* __restrict__ w1,
                                                         const float* __restrict__ b1, const float* __restrict__ g,
                                                         const float* __restrict__ be, int d, float* __restrict__ hsum,
                                                         int64_t ld, const int64_t* __restrict__ rows_dev) {
    if (rows_dev) rows = min(rows, *rows_dev);
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float wx[KC], wy[KC], bb[KC], gg[KC], bt[KC];
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        const int c = lane + 32 * k;
        const bool ok = c < d;
        wx[k] = ok ? w1[2 * c] : 0.f;
        wy[k] = ok ? w1[2 * c + 1] : 0.f;
        bb[k] = ok ? b1[c] : 0.f;
        gg[k] = ok ? g[c] : 0.f;
        bt[k] = ok ? be[c] : 0.f;
    }
    const float inv_d = 1.0f / (float)d;
    for (int64_t r = warp; r < rows; r += nwarps) {
        const int64_t s = row0 + r;
        const float x = __ldg(pa + s), y = __ldg(pb + s);
        float z1[KC], z2[KC];
        float s1 = 0.f, s2 = 0.f;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            z1[k] = fmaf(wx[k], x, fmaf(wy[k], y, bb[k]));
            z2[k] = fmaf(wx[k], y, fmaf(wy[k], x, bb[k]));
            s1 += z1[k];  // padded channels contribute exactly 0
            s2 += z2[k];
        }
        const float m1 = warp_sum(s1) * inv_d, m2 = warp_sum(s2) * inv_d;
        float v1 = 0.f, v2 = 0.f;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const bool ok = lane + 32 * k < d;
            const float d1 = ok ? z1[k] - m1 : 0.f, d2 = ok ? z2[k] - m2 : 0.f;
            v1 = fmaf(d1, d1, v1);
            v2 = fmaf(d2, d2, v2);
        }
        const float r1 = rsqrtf(warp_sum(v1) * inv_d + 1e-5f), r2 = rsqrtf(warp_sum(v2) * inv_d + 1e-5f);
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const int c = lane + 32 * k;
            if (c < d) {
                const float h1 = fmaxf(fmaf((z1[k] - m1) * r1, gg[k], bt[k]), 0.f);
                const float h2 = fmaxf(fmaf((z2[k] - m2) * r2, gg[k], bt[k]), 0.f);
                hsum[s * ld + c] = h1 + h2;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// fp32 contraction C = epi(A W^T + bias): 64x64 tile, BK 16, 4x4 register micro-tile.
// (First-correct SIMT path; the tcgen05 kernel in gemm_tc.cu takes the large aligned shapes.)
// ---------------------------------------------------------------------------------------
constexpr int BM = 64, BN = 64, BK = 16;

__global__ void __launch_bounds__(256) gemm_simt_kernel(const float* __restrict__ A, int64_t lda,
                                                        const float* __restrict__ W, int64_t ldw,
                                                        const float* __restrict__ bias, float bias_scale,
                                                        float* __restrict__ C, int64_t ldc, int64_t M, int N, int K,
                                                        int epi) {
    __shared__ float As[BK][BM + 4];
    __shared__ float Ws[BK][BN + 4];
    const int tid = threadIdx.x;
    const int64_t m0 = (int64_t)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;
    const int tx = tid & 15, ty = tid >> 4;  // 16 x 16 threads, each 4 (m) x 4 (n)
    float acc[4][4] = {};
    // loader mapping: 64 rows x 16 k = 1024 elements, 4 per thread: row = tid/4, k = (tid%4)*4..+3
    const int lr = tid >> 2, lk = (tid & 3) * 4;
    for (int k0 = 0; k0 < K; k0 += BK) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int k = k0 + lk + q;
            const int64_t m = m0 + lr;
            const int n = n0 + lr;
            As[lk + q][lr] = (m < M && k < K) ? __ldg(A + m * lda + k) : 0.f;
            Ws[lk + q][lr] = (n < N && k < K) ? __ldg(W + (int64_t)n * ldw + k) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[4], w[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                a[q] = As[k][ty * 4 + q];
                w[q] = Ws[k][tx * 4 + q];
            }
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], w[c], acc[r][c]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int64_t m = m0 + ty * 4 + r;
        if (m >= M) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int n = n0 + tx * 4 + c;
            if (n >= N) continue;
            float v = acc[r][c];
            if (bias) v += bias_scale * __ldg(bias + n);
            if (epi == LPF_EPI_RELU) v = fmaxf(v, 0.f);
            else if (epi == LPF_EPI_SIGMOID) v = 1.0f / (1.0f + expf(-v));
            C[m * ldc + n] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Row-wise LayerNorm (+ReLU, +residual); one warp per row, two-pass statistics.
// ---------------------------------------------------------------------------------------
// DROP: dropout after the activation, before the residual (the GCN epilogue of lpf_gcn_layer_dropout); mask row =
// row0 + r, column = c (rule in common.cuh)
template <bool DROP>
__global__ void __launch_bounds__(256) layernorm_act_kernel(const float* X, int64_t ldx,
                                                            const float* __restrict__ g, const float* __restrict__ b,
                                                            const float* R, int64_t ldr,
                                                            float* Y, int64_t ldy, int64_t rows, int n,
                                                            int relu, const int64_t* __restrict__ rows_dev,
                                                            int64_t row0, const uint64_t* seed_p, int site, uint64_t thr,
                                                            float scale) {
    if (rows_dev) rows = min(rows, *rows_dev);
    uint64_t seed = 0;
    if constexpr (DROP) seed = *seed_p;
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const float inv_n = 1.0f / (float)n;
    for (int64_t r = warp; r < rows; r += nwarps) {
        const float* x = X + r * ldx;
        float mean = 0.f, rstd = 1.f;
        if (g) {
            float s = 0.f;
            for (int c = lane; c < n; c += 32) s += x[c];
            mean = warp_sum(s) * inv_n;
            float v = 0.f;
            for (int c = lane; c < n; c += 32) {
                const float dlt = x[c] - mean;
                v = fmaf(dlt, dlt, v);
            }
            rstd = rsqrtf(warp_sum(v) * inv_n + 1e-5f);
        }
        for (int c = lane; c < n; c += 32) {
            float y = g ? fmaf((x[c] - mean) * rstd, __ldg(g + c), __ldg(b + c)) : x[c];
            if (relu) y = fmaxf(y, 0.f);
            if constexpr (DROP) y = dropout_apply(y, uint4_word(dropout_bits(seed, site, row0 + r, c >> 2), c & 3), thr, scale);
            if (R) y += R[r * ldr + c];
            Y[r * ldy + c] = y;
        }
    }
}

// ---------------------------------------------------------------------------------------
// Link gathers: xsum = X[a]+X[b], xprod = X[a]*X[b]
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_links_kernel(const int64_t* __restrict__ links, int64_t bs,
                                                           const int32_t* __restrict__ idx, int64_t n,
                                                           const float* __restrict__ X, int64_t ldx, int d,
                                                           float* __restrict__ xsum, int64_t lds,
                                                           float* __restrict__ xprod, int64_t ldp,
                                                           const int64_t* __restrict__ n_dev, int x_bf16) {
    if (n_dev) n = min(n, *n_dev);
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const bool vec = !x_bf16 && (d % 4 == 0) && (ldx % 4 == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) &&
                     (!xsum || ((lds % 4 == 0) && (reinterpret_cast<uintptr_t>(xsum) & 15) == 0)) &&
                     (!xprod || ((ldp % 4 == 0) && (reinterpret_cast<uintptr_t>(xprod) & 15) == 0));
    for (int64_t i = warp; i < n; i += nwarps) {
        const int64_t pos = idx ? (int64_t)__ldg(idx + i) : i;
        const int64_t a = __ldg(links + pos), b = __ldg(links + bs + pos);
        const float* xa = X + a * ldx;
        const float* xb = X + b * ldx;
        if (vec) {
            for (int c = lane * 4; c < d; c += 128) {
                const float4 u = __ldg(reinterpret_cast<const float4*>(xa + c));
                const float4 w = __ldg(reinterpret_cast<const float4*>(xb + c));
                if (xsum) *reinterpret_cast<float4*>(xsum + i * lds + c) = make_float4(u.x + w.x, u.y + w.y, u.z + w.z, u.w + w.w);
                if (xprod) *reinterpret_cast<float4*>(xprod + i * ldp + c) = make_float4(u.x * w.x, u.y * w.y, u.z * w.z, u.w * w.w);
            }
        } else {
            const uint16_t* ha = reinterpret_cast<const uint16_t*>(X) + a * ldx;      // (bf16 table: same row, 2-byte elements)
            const uint16_t* hb = reinterpret_cast<const uint16_t*>(X) + b * ldx;
            for (int c = lane; c < d; c += 32) {
                const float u = x_bf16 ? __uint_as_float((uint32_t)__ldg(ha + c) << 16) : __ldg(xa + c);
                const float w = x_bf16 ? __uint_as_float((uint32_t)__ldg(hb + c) << 16) : __ldg(xb + c);
                if (xsum) xsum[i * lds + c] = u + w;
                if (xprod) xprod[i * ldp + c] = u * w;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// Query groups -> link pairs: links[0, i] = source[(j0 + i) / K], links[1, i] = targets[i] for the flat range
// i < n of the grouped form (flat index q K + j, the order of the reference's source.repeat(K) x targets).  An id
// outside [0, num_nodes) is written as 0, so no later kernel reads out of bounds, and raises *bad.
// ---------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) expand_query_links_kernel(const T* __restrict__ source,
                                                                 const T* __restrict__ targets, int64_t K, int64_t j0,
                                                                 int64_t n, int64_t num_nodes,
                                                                 int64_t* __restrict__ links, int64_t ld,
                                                                 int64_t* __restrict__ bad) {
    bool flag = false;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = (int64_t)__ldg(targets + i);
        const int64_t s = (int64_t)__ldg(source + (j0 + i) / K);     // (consecutive threads: the same cached word)
        const bool s_ok = s >= 0 && s < num_nodes, t_ok = t >= 0 && t < num_nodes;
        links[i] = s_ok ? s : 0;
        links[ld + i] = t_ok ? t : 0;
        flag |= !(s_ok && t_ok);
    }
    if (__any_sync(0xffffffffu, flag) && (threadIdx.x & 31) == 0) *bad = 1;
}

// dst[r,:] = fill[:] for every row / dst[idx[j],:] = src[j,:]
__global__ void __launch_bounds__(256) fill_rows_kernel(float* __restrict__ dst, int64_t ldd, int64_t rows, int d,
                                                        const float* __restrict__ fill) {
    const int64_t total = rows * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / d;
        const int c = (int)(e - r * d);
        dst[r * ldd + c] = __ldg(fill + c);
    }
}
__global__ void __launch_bounds__(256) scatter_rows_kernel(const float* __restrict__ src, int64_t lds,
                                                           const int32_t* __restrict__ idx, int64_t n,
                                                           float* __restrict__ dst, int64_t ldd, int d) {
    const int64_t total = n * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = e / d;
        const int c = (int)(e - j * d);
        dst[(int64_t)__ldg(idx + j) * ldd + c] = src[j * lds + c];
    }
}

static inline unsigned warp_grid(int64_t items, int threads) {
    const int wpb = threads / 32;
    int64_t blocks = (items + wpb - 1) / wpb;
    const int64_t cap = (int64_t)kNumSMs * 8 * 2;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}

}  // namespace lpf

using namespace lpf;

extern "C" int lpf_rpe_hidden(const float* src_ppr, const float* tgt_ppr, int64_t row0, int64_t rows, const float* w1,
                              const float* b1, const float* ln_w, const float* ln_b, int32_t d, float* hsum,
                              int64_t ld_hsum, const int64_t* rows_dev, void* stream) {
    LPF_REQUIRE(rows >= 0 && row0 >= 0, "negative row range");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(src_ppr && tgt_ppr && w1 && b1 && ln_w && ln_b && hsum, "NULL argument");
    LPF_REQUIRE(d >= 1 && d <= 512, "d must be in [1,512]");
    LPF_REQUIRE(ld_hsum >= d, "ld_hsum < d");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = warp_grid(rows, 256);
    const int kc = (d + 31) / 32;
#define LPF_RPE(KC) rpe_hidden_kernel<KC><<<grid, 256, 0, st>>>(src_ppr, tgt_ppr, row0, rows, w1, b1, ln_w, ln_b, d, hsum, ld_hsum, rows_dev)
    if (kc <= 1) LPF_RPE(1);
    else if (kc <= 2) LPF_RPE(2);
    else if (kc <= 4) LPF_RPE(4);
    else if (kc <= 8) LPF_RPE(8);
    else LPF_RPE(16);
#undef LPF_RPE
    return check_launch("lpf_rpe_hidden");
}

namespace lpf {
int gemm_tc_try(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float bias_scale,
                float* C, int64_t ldc, int64_t M, int32_t N, int32_t K, int epilogue, cudaStream_t st);
}

extern "C" int lpf_gemm(const float* A, int64_t lda, const float* W, int64_t ldw, const float* bias, float bias_scale,
                        float* C, int64_t ldc, int64_t M, int32_t N, int32_t K, int epilogue, void* stream) {
    LPF_REQUIRE(M >= 0 && N >= 1 && K >= 1, "bad shape");
    if (M == 0) return LPF_OK;
    LPF_REQUIRE(A && W && C, "NULL argument");
    LPF_REQUIRE(lda >= K && ldw >= K && ldc >= N, "leading dimension too small");
    LPF_REQUIRE(epilogue >= LPF_EPI_NONE && epilogue <= LPF_EPI_SIGMOID, "bad epilogue");
    cudaStream_t st = (cudaStream_t)stream;
    const dim3 grid((unsigned)((M + BM - 1) / BM), (unsigned)((N + BN - 1) / BN));
    gemm_simt_kernel<<<grid, 256, 0, st>>>(A, lda, W, ldw, bias, bias_scale, C, ldc, M, N, K, epilogue);
    return check_launch("lpf_gemm");
}

extern "C" int lpf_layernorm_act(const float* X, int64_t ldx, const float* gamma, const float* beta,
                                 const float* residual, int64_t ldr, float* Y, int64_t ldy, int64_t rows, int32_t n,
                                 int relu, const int64_t* rows_dev, void* stream) {
    LPF_REQUIRE(rows >= 0 && n >= 1, "bad shape");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(X && Y, "NULL argument");
    LPF_REQUIRE((gamma == nullptr) == (beta == nullptr), "gamma and beta must both be given or both NULL");
    LPF_REQUIRE(ldx >= n && ldy >= n && (!residual || ldr >= n), "leading dimension too small");
    layernorm_act_kernel<false><<<warp_grid(rows, 256), 256, 0, (cudaStream_t)stream>>>(
        X, ldx, gamma, beta, residual, ldr, Y, ldy, rows, n, relu, rows_dev, 0, nullptr, 0, 0, 0.f);
    return check_launch("lpf_layernorm_act");
}

extern "C" int lpf_layernorm_act_dropout(const float* X, int64_t ldx, const float* gamma, const float* beta, int relu,
                                         int64_t row0, const uint64_t* seed, int32_t site, double p,
                                         const float* residual, int64_t ldr, float* Y, int64_t ldy, int64_t rows,
                                         int32_t n, void* stream) {
    uint64_t thr;
    float scale;
    LPF_REQUIRE(dropout_rule(p, &thr, &scale), "p must be in [0, 1]");
    LPF_REQUIRE(rows >= 0 && n >= 1 && row0 >= 0, "bad shape");
    LPF_REQUIRE(seed, "seed is NULL");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(X && Y, "NULL argument");
    LPF_REQUIRE((gamma == nullptr) == (beta == nullptr), "gamma and beta must both be given or both NULL");
    LPF_REQUIRE(ldx >= n && ldy >= n && (!residual || ldr >= n), "leading dimension too small");
    layernorm_act_kernel<true><<<warp_grid(rows, 256), 256, 0, (cudaStream_t)stream>>>(
        X, ldx, gamma, beta, residual, ldr, Y, ldy, rows, n, relu, nullptr, row0, seed, site, thr, scale);
    return check_launch("lpf_layernorm_act_dropout");
}

extern "C" int lpf_gather_links(const int64_t* links, int64_t bs, const int32_t* idx, int64_t n, const float* X,
                                int64_t ldx, int32_t d, float* xsum, int64_t ld_sum, float* xprod, int64_t ld_prod,
                                const int64_t* n_dev, int x_bf16, void* stream) {
    LPF_REQUIRE(bs >= 0 && n >= 0 && d >= 1, "bad shape");
    LPF_REQUIRE(idx || n == bs, "n must equal bs when idx is NULL");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(links && X, "NULL argument");
    LPF_REQUIRE(xsum || xprod, "no output requested");
    LPF_REQUIRE(ldx >= d && (!xsum || ld_sum >= d) && (!xprod || ld_prod >= d), "leading dimension too small");
    gather_links_kernel<<<warp_grid(n, 256), 256, 0, (cudaStream_t)stream>>>(links, bs, idx, n, X, ldx, d, xsum, ld_sum,
                                                                             xprod, ld_prod, n_dev, x_bf16);
    return check_launch("lpf_gather_links");
}

extern "C" int lpf_expand_query_links(const void* source, const void* targets, int32_t id_bytes, int64_t K, int64_t j0,
                                      int64_t n, int64_t num_nodes, int64_t* links, int64_t ld, int64_t* bad,
                                      void* stream) {
    LPF_REQUIRE(id_bytes == 4 || id_bytes == 8, "id_bytes must be 4 or 8");
    LPF_REQUIRE(K >= 1, "K must be >= 1");
    LPF_REQUIRE(n >= 0 && j0 >= 0 && j0 < K, "bad range (need n >= 0, 0 <= j0 < K)");
    LPF_REQUIRE(num_nodes >= 0, "num_nodes < 0");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(source && targets && links && bad, "NULL argument");
    LPF_REQUIRE(ld >= n, "ld < n");
    int64_t blocks = (n + 255) / 256;
    const int64_t cap = (int64_t)kNumSMs * 8;
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    if (id_bytes == 4)
        expand_query_links_kernel<int32_t><<<(unsigned)blocks, 256, 0, st>>>(
            (const int32_t*)source, (const int32_t*)targets, K, j0, n, num_nodes, links, ld, bad);
    else
        expand_query_links_kernel<int64_t><<<(unsigned)blocks, 256, 0, st>>>(
            (const int64_t*)source, (const int64_t*)targets, K, j0, n, num_nodes, links, ld, bad);
    return check_launch("lpf_expand_query_links");
}

extern "C" int lpf_scatter_rows(const float* src, int64_t ld_src, const int32_t* idx, int64_t n, float* dst,
                                int64_t ld_dst, int64_t rows, int32_t d, const float* fill_row, void* stream) {
    LPF_REQUIRE(n >= 0 && rows >= 0 && d >= 1, "bad shape");
    LPF_REQUIRE(rows == 0 || dst, "dst is NULL");
    LPF_REQUIRE(n == 0 || (src && idx), "src/idx is NULL");
    LPF_REQUIRE(ld_dst >= d && (n == 0 || ld_src >= d), "leading dimension too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cap = (int64_t)kNumSMs * 16;
    if (fill_row && rows > 0) {
        int64_t blocks = (rows * d + 255) / 256;
        fill_rows_kernel<<<(unsigned)(blocks > cap ? cap : blocks), 256, 0, st>>>(dst, ld_dst, rows, d, fill_row);
    }
    if (n > 0) {
        int64_t blocks = (n * d + 255) / 256;
        scatter_rows_kernel<<<(unsigned)(blocks > cap ? cap : blocks), 256, 0, st>>>(src, ld_src, idx, n, dst, ld_dst, d);
    }
    return check_launch("lpf_scatter_rows");
}
