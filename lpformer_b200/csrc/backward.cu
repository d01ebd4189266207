// Backward pass of the host-sized path: the gradients of every stage of LinkTransformer.forward / mlp_score with
// respect to the reference's own parameters and to X_node (autograd Functions in lpformer_b200/autograd.py).
//
// Every reduction over rows (links, pairs, nodes) that produces a parameter gradient is two-stage and deterministic:
// a fixed grid writes per-CTA partial sums into a caller-owned workspace, and one more launch adds them in CTA order.
// Scatters into node-indexed tables (dX of the link gathers, dKV of the attention) use fp32 atomics.
#include "common.cuh"

namespace lpf {

constexpr int kBwdThreads = 256;
constexpr int kBwdWarps = kBwdThreads / 32;
constexpr int kBwdMaxBlocks = kNumSMs * 4;

static inline unsigned bwd_grid(int64_t warps_of_work) {
    int64_t b = (warps_of_work + kBwdWarps - 1) / kBwdWarps;
    if (b > kBwdMaxBlocks) b = kBwdMaxBlocks;
    if (b < 1) b = 1;
    return (unsigned)b;
}

// out[c] (+)= sum_b part[b * stride + c] for c < n, b in CTA order
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ part, int64_t blocks, int64_t stride,
                                                              int64_t n, float* __restrict__ out, int accumulate) {
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n; c += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int64_t b = 0; b < blocks; ++b) s += part[b * stride + c];
        out[c] = accumulate ? out[c] + s : s;
    }
}

static void launch_reduce(const float* part, int64_t blocks, int64_t stride, int64_t n, float* out, int accumulate,
                          cudaStream_t st) {
    int64_t g = (n + 255) / 256;
    if (g > kBwdMaxBlocks) g = kBwdMaxBlocks;
    reduce_partials_kernel<<<(unsigned)(g < 1 ? 1 : g), 256, 0, st>>>(part, blocks, stride, n, out, accumulate);
}

// ---------------------------------------------------------------------------------------
// LayerNorm (+ReLU) backward, one warp per row, statistics recomputed from the saved pre-norm row x:
//   xh = (x - mean) rstd,  z = xh g + b,  dz = dy [z > 0],  dx = rstd (dz g - mean(dz g) - xh mean(dz g xh)),
//   dg += dz xh,  db += dz.   Without g: dx = dy [x > 0] (ReLU only) or dy.
// Each warp keeps its own dg / db row in shared memory; the CTA's rows are summed into its partial.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBwdThreads) ln_act_bwd_kernel(const float* __restrict__ X, int64_t ldx,
                                                                 const float* __restrict__ g, const float* __restrict__ b,
                                                                 int relu, const float* __restrict__ dY, int64_t lddy,
                                                                 float* dX, int64_t lddx, int acc_dx, int64_t rows, int n,
                                                                 float* __restrict__ part) {
    extern __shared__ float s_param[];      // [kBwdWarps][2n]  (only with g)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t gw = (int64_t)blockIdx.x * kBwdWarps + warp, nw = (int64_t)gridDim.x * kBwdWarps;
    const float inv_n = 1.0f / (float)n;
    float* my = g ? s_param + (size_t)warp * 2 * n : nullptr;
    if (g)
        for (int c = lane; c < 2 * n; c += 32) my[c] = 0.f;
    __syncwarp();                           // (my[n + c] is zeroed by another lane than the one that adds to it)
    for (int64_t r = gw; r < rows; r += nw) {
        const float* x = X + r * ldx;
        const float* dy = dY + r * lddy;
        float* dx = dX + r * lddx;
        if (!g) {
            for (int c = lane; c < n; c += 32) {
                float v = dy[c];
                if (relu && !(x[c] > 0.f)) v = 0.f;
                dx[c] = acc_dx ? dx[c] + v : v;
            }
            continue;
        }
        float s = 0.f;
        for (int c = lane; c < n; c += 32) s += x[c];
        const float mean = warp_sum(s) * inv_n;
        float v = 0.f;
        for (int c = lane; c < n; c += 32) {
            const float dl = x[c] - mean;
            v = fmaf(dl, dl, v);
        }
        const float rstd = rsqrtf(warp_sum(v) * inv_n + 1e-5f);
        float s1 = 0.f, s2 = 0.f;
        for (int c = lane; c < n; c += 32) {
            const float xh = (x[c] - mean) * rstd;
            float dz = dy[c];
            if (relu && !(fmaf(xh, __ldg(g + c), __ldg(b + c)) > 0.f)) dz = 0.f;
            my[c] += dz * xh;
            my[n + c] += dz;
            const float dg = dz * __ldg(g + c);
            s1 += dg;
            s2 = fmaf(dg, xh, s2);
        }
        s1 = warp_sum(s1) * inv_n;
        s2 = warp_sum(s2) * inv_n;
        for (int c = lane; c < n; c += 32) {
            const float xh = (x[c] - mean) * rstd;
            float dz = dy[c];
            if (relu && !(fmaf(xh, __ldg(g + c), __ldg(b + c)) > 0.f)) dz = 0.f;
            const float val = rstd * (dz * __ldg(g + c) - s1 - xh * s2);
            dx[c] = acc_dx ? dx[c] + val : val;
        }
    }
    if (!g) return;
    __syncthreads();
    for (int c = threadIdx.x; c < 2 * n; c += kBwdThreads) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += s_param[(size_t)w * 2 * n + c];
        part[(int64_t)blockIdx.x * 2 * n + c] = t;
    }
}

// ---------------------------------------------------------------------------------------
// Weight gradient dW[N,K] (+)= dY[M,N]^T A[M,K], db[N] (+)= sum_m dY[m,:]: the M rows are split over gridDim.z slices,
// each CTA a 64 (n) x 64 (k) tile of one slice (fp32 FFMA, 4x4 register micro-tile, 16 rows per shared-memory stage),
// partials [slice][N*K + N] reduced in slice order.
// ---------------------------------------------------------------------------------------
constexpr int WG_T = 64, WG_BM = 16;

__global__ void __launch_bounds__(256) wgrad_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ dY,
                                                    int64_t lddy, int64_t M, int N, int K, int64_t chunk,
                                                    float* __restrict__ part) {
    __shared__ float Ys[WG_BM][WG_T + 4];
    __shared__ float As[WG_BM][WG_T + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;     // ty: 4 rows of n, tx: 4 columns of k
    const int n0 = blockIdx.y * WG_T, k0 = blockIdx.x * WG_T;
    const int64_t m_lo = (int64_t)blockIdx.z * chunk, m_hi = min(M, m_lo + chunk);
    const int64_t slot = (int64_t)N * K + N;
    float acc[4][4] = {}, bsum[4] = {};
    const bool want_b = blockIdx.x == 0;
    const int lr = tid >> 4, lc = (tid & 15) * 4;                   // loader: 16 rows x 64 columns, 4 per thread
    for (int64_t m0 = m_lo; m0 < m_hi; m0 += WG_BM) {
        const int64_t m = m0 + lr;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int n = n0 + lc + q, k = k0 + lc + q;
            Ys[lr][lc + q] = (m < m_hi && n < N) ? __ldg(dY + m * lddy + n) : 0.f;
            As[lr][lc + q] = (A && m < m_hi && k < K) ? __ldg(A + m * lda + k) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int mm = 0; mm < WG_BM; ++mm) {
            float y[4], a[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                y[q] = Ys[mm][ty * 4 + q];
                a[q] = As[mm][tx * 4 + q];
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(y[r], a[c], acc[r][c]);
                bsum[r] += y[r];
            }
        }
        __syncthreads();
    }
    float* out = part + (int64_t)blockIdx.z * slot;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int n = n0 + ty * 4 + r;
        if (n >= N) continue;
        if (A) {
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int k = k0 + tx * 4 + c;
                if (k < K) out[(int64_t)n * K + k] = acc[r][c];
            }
        }
        if (want_b && tx == 0) out[(int64_t)N * K + n] = bsum[r];
    }
}

// (dW, db) (+)= reduce over slices
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, int64_t slices, int N, int K,
                                                           float* dW, int64_t ldw, float* db, int accumulate) {
    const int64_t slot = (int64_t)N * K + N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < slot; e += (int64_t)gridDim.x * blockDim.x) {
        float* dst;
        if (e < (int64_t)N * K) {
            if (!dW) continue;
            dst = dW + (e / K) * ldw + (e % K);
        } else {
            if (!db) continue;
            dst = db + (e - (int64_t)N * K);
        }
        float s = 0.f;
        for (int64_t z = 0; z < slices; ++z) s += part[z * slot + e];
        *dst = accumulate ? *dst + s : s;
    }
}

static int64_t wgrad_slices(int64_t M, int N, int K) {
    const int64_t tiles = (int64_t)((K + WG_T - 1) / WG_T) * ((N + WG_T - 1) / WG_T);
    int64_t s = (int64_t)kNumSMs * 8 / tiles;
    const int64_t by_rows = (M + 255) / 256;          // at least 256 rows per slice
    if (s > by_rows) s = by_rows;
    if (s > 65535) s = 65535;
    return s < 1 ? 1 : s;
}

// ---------------------------------------------------------------------------------------
// Elementwise activation backward from the saved output: ReLU dx = dy [y > 0], sigmoid dx = dy y (1 - y).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) act_bwd_kernel(const float* __restrict__ Y, int64_t ldy, const float* __restrict__ dY,
                                                      int64_t lddy, float* __restrict__ dX, int64_t lddx, int64_t rows, int n,
                                                      int act) {
    const int64_t total = rows * n;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / n;
        const int c = (int)(e - r * n);
        const float y = Y[r * ldy + c], g = dY[r * lddy + c];
        dX[r * lddx + c] = act == LPF_EPI_SIGMOID ? g * y * (1.f - y) : (y > 0.f ? g : 0.f);
    }
}

// ---------------------------------------------------------------------------------------
// Link gathers backward: xsum = X[a] + X[b], xprod = X[a] * X[b]  ->  dX[a] += dsum + dprod X[b], dX[b] += dsum + dprod X[a]
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gather_links_bwd_kernel(const int64_t* __restrict__ links, int64_t bs,
                                                               const int32_t* __restrict__ idx, int64_t n,
                                                               const float* __restrict__ X, int64_t ldx, int d,
                                                               const float* __restrict__ dsum, int64_t lds,
                                                               const float* __restrict__ dprod, int64_t ldp,
                                                               float* __restrict__ dX, int64_t lddx) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < n; i += nwarps) {
        const int64_t pos = idx ? (int64_t)__ldg(idx + i) : i;
        const int64_t a = __ldg(links + pos), b = __ldg(links + bs + pos);
        for (int c = lane; c < d; c += 32) {
            float ga = dsum ? __ldg(dsum + i * lds + c) : 0.f, gb = ga;
            if (dprod) {
                const float gp = __ldg(dprod + i * ldp + c);
                ga = fmaf(gp, __ldg(X + b * ldx + c), ga);
                gb = fmaf(gp, __ldg(X + a * ldx + c), gb);
            }
            atomicAdd(dX + a * lddx + c, ga);
            atomicAdd(dX + b * lddx + c, gb);
        }
    }
}

// ---------------------------------------------------------------------------------------
// scatter_rows backward: dsrc[j] = dG[idx[j]];  dfill = sum of the rows of dG that idx does not name
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) scatter_rows_bwd_gather_kernel(const float* __restrict__ dG, int64_t ldg,
                                                                      const int32_t* __restrict__ idx, int64_t n, int d,
                                                                      float* __restrict__ dsrc, int64_t ld_src,
                                                                      uint8_t* __restrict__ mark) {
    const int64_t total = n * d;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = e / d;
        const int c = (int)(e - j * d);
        const int64_t r = __ldg(idx + j);
        if (dsrc) dsrc[j * ld_src + c] = dG[r * ldg + c];
        if (c == 0 && mark) mark[r] = 1;
    }
}

__global__ void __launch_bounds__(kBwdThreads) masked_colsum_kernel(const float* __restrict__ dG, int64_t ldg, int64_t rows,
                                                                    int d, const uint8_t* __restrict__ mark,
                                                                    float* __restrict__ part) {
    extern __shared__ float s_col[];        // [kBwdWarps][d]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* my = s_col + (size_t)warp * d;
    for (int c = lane; c < d; c += 32) my[c] = 0.f;
    for (int64_t r = (int64_t)blockIdx.x * kBwdWarps + warp; r < rows; r += (int64_t)gridDim.x * kBwdWarps) {
        if (mark && mark[r]) continue;
        for (int c = lane; c < d; c += 32) my[c] += dG[r * ldg + c];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < d; c += kBwdThreads) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += s_col[(size_t)w * d + c];
        part[(int64_t)blockIdx.x * d + c] = t;
    }
}

// ---------------------------------------------------------------------------------------
// RPE hidden backward (get_pos_encodings, reference models/link_transformer.py:182-211, first Linear + LayerNorm + ReLU
// of the PPR encoder MLP): per pair, for both orderings (x, y) = (pa, pb) and (pb, pa) — hsum = h(pa,pb) + h(pb,pa), so
// both see the same upstream dh — recompute z = W1 [x, y] + b1, its LayerNorm and ReLU, and accumulate
// dW1[:, 0] += dz x, dW1[:, 1] += dz y, db1 += dz, dg += dpre zh, dbeta += dpre.  One warp per pair, channels over lanes,
// the five accumulators in registers; per-CTA partials [5d] (w1x | w1y | b1 | g | beta).
// ---------------------------------------------------------------------------------------
template <int KC>
__global__ void __launch_bounds__(kBwdThreads) rpe_hidden_bwd_kernel(const float* __restrict__ pa, const float* __restrict__ pb,
                                                                     int64_t row0, int64_t rows, const float* __restrict__ w1,
                                                                     const float* __restrict__ b1, const float* __restrict__ g,
                                                                     const float* __restrict__ be, int d,
                                                                     const float* __restrict__ dh, int64_t ld_dh,
                                                                     float* __restrict__ part) {
    __shared__ float s_acc[kBwdWarps][5][KC * 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float wx[KC], wy[KC], bb[KC], gg[KC], bt[KC];
    float awx[KC], awy[KC], ab[KC], ag[KC], abt[KC];
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        const int c = lane + 32 * k;
        const bool ok = c < d;
        wx[k] = ok ? w1[2 * c] : 0.f;
        wy[k] = ok ? w1[2 * c + 1] : 0.f;
        bb[k] = ok ? b1[c] : 0.f;
        gg[k] = ok ? g[c] : 0.f;
        bt[k] = ok ? be[c] : 0.f;
        awx[k] = awy[k] = ab[k] = ag[k] = abt[k] = 0.f;
    }
    const float inv_d = 1.0f / (float)d;
    for (int64_t r = (int64_t)blockIdx.x * kBwdWarps + warp; r < rows; r += (int64_t)gridDim.x * kBwdWarps) {
        const int64_t s = row0 + r;
        const float p0 = __ldg(pa + s), p1 = __ldg(pb + s);
        float gd[KC];
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const int c = lane + 32 * k;
            gd[k] = c < d ? __ldg(dh + r * ld_dh + c) : 0.f;
        }
#pragma unroll
        for (int o = 0; o < 2; ++o) {
            const float x = o ? p1 : p0, y = o ? p0 : p1;
            float z[KC], sm = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                z[k] = fmaf(wx[k], x, fmaf(wy[k], y, bb[k]));
                sm += z[k];                     // (padded channels: exactly 0)
            }
            const float mean = warp_sum(sm) * inv_d;
            float v = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const float dl = lane + 32 * k < d ? z[k] - mean : 0.f;
                v = fmaf(dl, dl, v);
            }
            const float rstd = rsqrtf(warp_sum(v) * inv_d + 1e-5f);
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const bool ok = lane + 32 * k < d;
                const float zh = ok ? (z[k] - mean) * rstd : 0.f;
                const float pre = fmaf(zh, gg[k], bt[k]);
                const float dp = (ok && pre > 0.f) ? gd[k] : 0.f;
                ag[k] = fmaf(dp, zh, ag[k]);
                abt[k] += dp;
                const float dzh = dp * gg[k];
                s1 += dzh;
                s2 = fmaf(dzh, zh, s2);
                z[k] = zh;                       // (keep zh)
            }
            s1 = warp_sum(s1) * inv_d;
            s2 = warp_sum(s2) * inv_d;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const bool ok = lane + 32 * k < d;
                const float pre = fmaf(z[k], gg[k], bt[k]);
                const float dp = (ok && pre > 0.f) ? gd[k] : 0.f;
                const float dz = ok ? rstd * (dp * gg[k] - s1 - z[k] * s2) : 0.f;
                awx[k] = fmaf(dz, x, awx[k]);
                awy[k] = fmaf(dz, y, awy[k]);
                ab[k] += dz;
            }
        }
    }
#pragma unroll
    for (int k = 0; k < KC; ++k) {
        s_acc[warp][0][k * 32 + lane] = awx[k];
        s_acc[warp][1][k * 32 + lane] = awy[k];
        s_acc[warp][2][k * 32 + lane] = ab[k];
        s_acc[warp][3][k * 32 + lane] = ag[k];
        s_acc[warp][4][k * 32 + lane] = abt[k];
    }
    __syncthreads();
    for (int e = threadIdx.x; e < 5 * d; e += kBwdThreads) {
        const int f = e / d, c = e - f * d;
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < kBwdWarps; ++w) t += s_acc[w][f][c];
        part[(int64_t)blockIdx.x * 5 * d + e] = t;
    }
}

// partials [blocks][5d] -> dw1 [d, 2] (interleaved), db1, dg, dbeta
__global__ void __launch_bounds__(256) rpe_reduce_kernel(const float* __restrict__ part, int64_t blocks, int d,
                                                         float* dw1, float* db1, float* dg, float* dbe, int accumulate) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < 5 * d; e += gridDim.x * blockDim.x) {
        const int f = e / d, c = e - f * d;
        float s = 0.f;
        for (int64_t b = 0; b < blocks; ++b) s += part[b * 5 * d + e];
        float* dst = f == 0 ? dw1 + 2 * c : f == 1 ? dw1 + 2 * c + 1 : f == 2 ? db1 + c : f == 3 ? dg + c : dbe + c;
        *dst = accumulate ? *dst + s : s;
    }
}

// ---------------------------------------------------------------------------------------
// Attention backward (LinkTransformerLayer.forward + LinkAttention.forward / message, reference modules/layers.py:39-82,
// :161-224, in the algebra of attend.cu):
//   v_s = KV[u_s] + R_s,  sc_{s,h} = sum_c att[h,c] lrelu(v_s[h,c] q[h,c]),  alpha = segment softmax,
//   o = sum_s alpha_s v_s + bias,  y = LN(o).
// One warp per link.  Pass 1 recomputes the softmax state (max, sum, weighted sum) as the forward does; then
//   d_o = LN backward of dy;  gam_h = sum_c d_o (o - bias)  (= sum_s alpha_s dalpha_s);
// pass 2, per pair: dalpha_{s,h} = d_o[h] . v_s[h],  dsc = alpha (dalpha - gam),  dv = alpha d_o + dsc att lrelu'(v q) q,
//   dq += dsc att lrelu'(v q) v,  datt += dsc lrelu(v q);  dv goes to dR_s (or, through the row map, to the shared row
//   of its type) and is added into dKV[u_s].  Per link it writes dQ and one row of [d_o | dy xh | dy | datt] whose column
//   sums are the gradients of (bias, post_att_norm.weight, post_att_norm.bias, att).
// ---------------------------------------------------------------------------------------
struct AttendBwdParams {
    const int64_t* ptr;
    int64_t bs;
    const int32_t* idx;
    int64_t n;
    const int32_t* node;
    const float* KV;
    int64_t ld_kv;
    const float* R;
    int64_t ld_r;
    const int32_t* r_map;
    const float* r_const;
    const float* Q;
    int64_t ld_q;
    const float *att, *bias, *ln_w, *ln_b;
    const float* dY;
    int64_t ld_dy;
    float* dR;
    int64_t ld_dr;
    float* dR_const;      // [3][HC], accumulated
    float* dQ;
    int64_t ld_dq;
    float* dKV;
    int64_t ld_dkv;
    float* link_rows;     // [n][4 HC]
    int ch;
};

template <int H, int KC>
__global__ void __launch_bounds__(kBwdThreads, 1) attend_bwd_kernel(const __grid_constant__ AttendBwdParams p) {
    const int lane = threadIdx.x & 31;
    const int C = p.ch, HC = H * C;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    float att[H][KC];
#pragma unroll
    for (int h = 0; h < H; ++h)
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const int c = lane + 32 * k;
            att[h][k] = c < C ? __ldg(p.att + h * C + c) : 0.f;
        }
    for (int64_t j = gw; j < p.n; j += nw) {
        const int64_t i = p.idx ? (int64_t)__ldg(p.idx + j) : j;
        float q[H][KC], acc[H][KC], mx[H], den[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            mx[h] = -INFINITY;
            den[h] = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const int c = lane + 32 * k;
                q[h][k] = c < C ? __ldg(p.Q + j * p.ld_q + h * C + c) : 0.f;
                acc[h][k] = 0.f;
            }
        }
        auto load_v = [&](int64_t s, float (&v)[H][KC]) {
            const int64_t u = __ldg(p.node + s);
            const float* rr = p.R + s * p.ld_r;
            if (p.r_map) {
                const int ri = __ldg(p.r_map + s);
                rr = ri >= 0 ? p.R + (int64_t)ri * p.ld_r : p.r_const + (int64_t)(-1 - ri) * HC;
            }
#pragma unroll
            for (int h = 0; h < H; ++h)
#pragma unroll
                for (int k = 0; k < KC; ++k) {
                    const int c = lane + 32 * k;
                    v[h][k] = c < C ? __ldg(p.KV + u * p.ld_kv + h * C + c) + __ldg(rr + h * C + c) : 0.f;
                }
        };
        auto score = [&](const float (&v)[H][KC], float (&sc)[H]) {
#pragma unroll
            for (int h = 0; h < H; ++h) {
                float part = 0.f;
#pragma unroll
                for (int k = 0; k < KC; ++k) {
                    float x = v[h][k] * q[h][k];
                    x = x > 0.f ? x : 0.2f * x;
                    part = fmaf(att[h][k], x, part);
                }
                sc[h] = warp_sum(part);
            }
        };
        // pass 1: softmax state
#pragma unroll 1
        for (int t = 0; t < 3; ++t)
            for (int64_t s = __ldg(p.ptr + t * p.bs + i), e = __ldg(p.ptr + t * p.bs + i + 1); s < e; ++s) {
                float v[H][KC], sc[H];
                load_v(s, v);
                score(v, sc);
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float m_new = fmaxf(mx[h], sc[h]);
                    const float scale = expf(mx[h] - m_new), w = expf(sc[h] - m_new);
                    den[h] = fmaf(den[h], scale, w);
#pragma unroll
                    for (int k = 0; k < KC; ++k) acc[h][k] = fmaf(w, v[h][k], acc[h][k] * scale);
                    mx[h] = m_new;
                }
            }
        // LayerNorm backward of y = LN(o)
        float o[H][KC], dy[H][KC], sum = 0.f;
#pragma unroll
        for (int h = 0; h < H; ++h) {
            const float inv = 1.0f / (den[h] + 1e-16f);
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const int c = lane + 32 * k;
                acc[h][k] *= inv;                                  // acc = o - bias
                o[h][k] = c < C ? acc[h][k] + __ldg(p.bias + h * C + c) : 0.f;
                dy[h][k] = c < C ? __ldg(p.dY + j * p.ld_dy + h * C + c) : 0.f;
                sum += o[h][k];
            }
        }
        const float mean = warp_sum(sum) / (float)HC;
        float var = 0.f;
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const float dl = lane + 32 * k < C ? o[h][k] - mean : 0.f;
                var = fmaf(dl, dl, var);
            }
        const float rstd = rsqrtf(warp_sum(var) / (float)HC + 1e-5f);
        float s1 = 0.f, s2 = 0.f;
        float* lrow = p.link_rows + j * 4 * HC;
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const int c = lane + 32 * k;
                const float xh = (o[h][k] - mean) * rstd;
                o[h][k] = xh;
                if (c < C) {
                    lrow[HC + h * C + c] = dy[h][k] * xh;
                    lrow[2 * HC + h * C + c] = dy[h][k];
                }
                const float dg = c < C ? dy[h][k] * __ldg(p.ln_w + h * C + c) : 0.f;
                dy[h][k] = dg;
                s1 += dg;
                s2 = fmaf(dg, xh, s2);
            }
        s1 = warp_sum(s1) / (float)HC;
        s2 = warp_sum(s2) / (float)HC;
        float gam[H];
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float part = 0.f;
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const int c = lane + 32 * k;
                dy[h][k] = c < C ? rstd * (dy[h][k] - s1 - o[h][k] * s2) : 0.f;      // dy := d_o
                if (c < C) lrow[h * C + c] = dy[h][k];
                part = fmaf(dy[h][k], acc[h][k], part);
            }
            gam[h] = warp_sum(part);
        }
        // pass 2: per pair (acc := dq, o := datt)
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int k = 0; k < KC; ++k) acc[h][k] = o[h][k] = 0.f;
#pragma unroll 1
        for (int t = 0; t < 3; ++t) {
            float rc[H][KC];
            bool any_const = false;
#pragma unroll
            for (int h = 0; h < H; ++h)
#pragma unroll
                for (int k = 0; k < KC; ++k) rc[h][k] = 0.f;
            for (int64_t s = __ldg(p.ptr + t * p.bs + i), e = __ldg(p.ptr + t * p.bs + i + 1); s < e; ++s) {
                float v[H][KC], sc[H];
                load_v(s, v);
                score(v, sc);
                float dv[H][KC];
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    const float alpha = expf(sc[h] - mx[h]) / (den[h] + 1e-16f);
                    float part = 0.f;
#pragma unroll
                    for (int k = 0; k < KC; ++k) part = fmaf(dy[h][k], v[h][k], part);
                    const float dsc = alpha * (warp_sum(part) - gam[h]);
#pragma unroll
                    for (int k = 0; k < KC; ++k) {
                        const float x = v[h][k] * q[h][k];
                        const float gx = dsc * att[h][k] * (x > 0.f ? 1.f : 0.2f);
                        o[h][k] = fmaf(dsc, x > 0.f ? x : 0.2f * x, o[h][k]);
                        acc[h][k] = fmaf(gx, v[h][k], acc[h][k]);
                        dv[h][k] = fmaf(alpha, dy[h][k], gx * q[h][k]);
                    }
                }
                const int64_t u = __ldg(p.node + s);
                int ri = 0;
                if (p.r_map) ri = __ldg(p.r_map + s);
                const int64_t rrow = p.r_map ? (int64_t)ri : s;
#pragma unroll
                for (int h = 0; h < H; ++h)
#pragma unroll
                    for (int k = 0; k < KC; ++k) {
                        const int c = lane + 32 * k;
                        if (c < C) {
                            atomicAdd(p.dKV + u * p.ld_dkv + h * C + c, dv[h][k]);
                            if (rrow >= 0) p.dR[rrow * p.ld_dr + h * C + c] = dv[h][k];
                            else rc[h][k] += dv[h][k];
                        }
                    }
                any_const |= rrow < 0;
            }
            if (any_const) {
#pragma unroll
                for (int h = 0; h < H; ++h)
#pragma unroll
                    for (int k = 0; k < KC; ++k) {
                        const int c = lane + 32 * k;
                        if (c < C) atomicAdd(p.dR_const + t * HC + h * C + c, rc[h][k]);
                    }
            }
        }
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int k = 0; k < KC; ++k) {
                const int c = lane + 32 * k;
                if (c < C) {
                    p.dQ[j * p.ld_dq + h * C + c] = acc[h][k];
                    lrow[3 * HC + h * C + c] = o[h][k];
                }
            }
    }
}

template <int H>
static int launch_attend_bwd(const AttendBwdParams& p, cudaStream_t st) {
    const int kc = (p.ch + 31) / 32;
    void (*kern)(const AttendBwdParams) = nullptr;
    if (kc <= 1) kern = attend_bwd_kernel<H, 1>;
    else if (kc <= 2) { if constexpr (H * 2 <= 16) kern = attend_bwd_kernel<H, 2>; }
    else if (kc <= 4) { if constexpr (H * 4 <= 16) kern = attend_bwd_kernel<H, 4>; }
    else if (kc <= 8) { if constexpr (H * 8 <= 16) kern = attend_bwd_kernel<H, 8>; }
    else { if constexpr (H * 16 <= 16) kern = attend_bwd_kernel<H, 16>; }
    if (!kern) {
        set_error("lpf_attend_backward: heads = %d, ch = %d not instantiated (heads*ceil(ch/32) <= 16)", H, p.ch);
        return LPF_ERR_UNSUPPORTED;
    }
    kern<<<bwd_grid(p.n), kBwdThreads, 0, st>>>(p);
    return check_launch("lpf_attend_backward");
}

}  // namespace lpf

using namespace lpf;

extern "C" int64_t lpf_layernorm_act_backward_workspace_bytes(int64_t rows, int32_t n) {
    if (rows < 0 || n < 1) return -1;
    return (int64_t)bwd_grid(rows) * 2 * n * (int64_t)sizeof(float);
}

extern "C" int lpf_layernorm_act_backward(const float* X, int64_t ldx, const float* gamma, const float* beta, int relu,
                                          const float* dY, int64_t lddy, float* dX, int64_t lddx, int accumulate_dx,
                                          float* dgamma, float* dbeta, int accumulate_param, int64_t rows, int32_t n,
                                          void* workspace, int64_t workspace_bytes, void* stream) {
    LPF_REQUIRE(rows >= 0 && n >= 1 && n <= 1024, "bad shape (1 <= n <= 1024)");
    LPF_REQUIRE((gamma == nullptr) == (beta == nullptr), "gamma and beta must both be given or both NULL");
    LPF_REQUIRE(ldx >= n && lddy >= n && lddx >= n, "leading dimension too small");
    cudaStream_t st = (cudaStream_t)stream;
    if (gamma) {
        LPF_REQUIRE(dgamma && dbeta, "dgamma / dbeta are NULL");
        LPF_REQUIRE(workspace && workspace_bytes >= lpf_layernorm_act_backward_workspace_bytes(rows, n), "workspace too small");
    }
    if (rows == 0) {
        if (gamma && !accumulate_param) {
            cudaMemsetAsync(dgamma, 0, (size_t)n * sizeof(float), st);
            cudaMemsetAsync(dbeta, 0, (size_t)n * sizeof(float), st);
        }
        return check_launch("lpf_layernorm_act_backward");
    }
    LPF_REQUIRE(X && dY && dX, "NULL argument");
    const unsigned grid = bwd_grid(rows);
    const size_t smem = gamma ? (size_t)kBwdWarps * 2 * n * sizeof(float) : 0;
    cudaError_t e = cudaFuncSetAttribute(ln_act_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(kBwdWarps * 2 * 1024 * sizeof(float)));
    if (e != cudaSuccess) {
        set_error("lpf_layernorm_act_backward: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return LPF_ERR_CUDA;
    }
    float* part = static_cast<float*>(workspace);
    ln_act_bwd_kernel<<<grid, kBwdThreads, smem, st>>>(X, ldx, gamma, beta, relu, dY, lddy, dX, lddx, accumulate_dx, rows, n,
                                                       part);
    if (gamma) {
        launch_reduce(part, grid, 2 * (int64_t)n, n, dgamma, accumulate_param, st);      // partial rows: [dgamma | dbeta]
        launch_reduce(part + n, grid, 2 * (int64_t)n, n, dbeta, accumulate_param, st);
    }
    return check_launch("lpf_layernorm_act_backward");
}

extern "C" int64_t lpf_gemm_wgrad_workspace_bytes(int64_t M, int32_t N, int32_t K) {
    if (M < 0 || N < 1 || K < 1) return -1;
    return wgrad_slices(M, N, K) * ((int64_t)N * K + N) * (int64_t)sizeof(float);
}

extern "C" int lpf_gemm_wgrad(const float* A, int64_t lda, const float* dY, int64_t lddy, int64_t M, int32_t N, int32_t K,
                              float* dW, int64_t ldw, float* db, int accumulate, void* workspace, int64_t workspace_bytes,
                              void* stream) {
    LPF_REQUIRE(M >= 0 && N >= 1 && K >= 1, "bad shape");
    LPF_REQUIRE(dW || db, "no output requested");
    LPF_REQUIRE(!dW || (A && ldw >= K && lda >= K), "dW needs A (lda >= K, ldw >= K)");
    LPF_REQUIRE(M == 0 || (dY && lddy >= N), "dY is NULL or lddy < N");
    LPF_REQUIRE(workspace && workspace_bytes >= lpf_gemm_wgrad_workspace_bytes(M, N, K), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t slices = wgrad_slices(M, N, K);
    int64_t chunk = (M + slices - 1) / slices;
    chunk = (chunk + WG_BM - 1) / WG_BM * WG_BM;
    float* part = static_cast<float*>(workspace);
    const dim3 grid(dW ? (unsigned)((K + WG_T - 1) / WG_T) : 1u, (unsigned)((N + WG_T - 1) / WG_T), (unsigned)slices);
    wgrad_kernel<<<grid, 256, 0, st>>>(dW ? A : nullptr, lda, dY, lddy, M, N, dW ? K : 1, chunk, part);
    const int Kp = dW ? K : 1;
    // (without dW the partial slots are [N * 1 + N]: only their db half is read)
    const int64_t slot = (int64_t)N * Kp + N;
    int64_t g = (slot + 255) / 256;
    if (g > kBwdMaxBlocks) g = kBwdMaxBlocks;
    wgrad_reduce_kernel<<<(unsigned)g, 256, 0, st>>>(part, slices, N, Kp, dW, ldw, db, accumulate);
    return check_launch("lpf_gemm_wgrad");
}

extern "C" int lpf_act_backward(const float* Y, int64_t ldy, const float* dY, int64_t lddy, float* dX, int64_t lddx,
                                int64_t rows, int32_t n, int act, void* stream) {
    LPF_REQUIRE(rows >= 0 && n >= 1, "bad shape");
    LPF_REQUIRE(act == LPF_EPI_RELU || act == LPF_EPI_SIGMOID, "act must be LPF_EPI_RELU or LPF_EPI_SIGMOID");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(Y && dY && dX, "NULL argument");
    LPF_REQUIRE(ldy >= n && lddy >= n && lddx >= n, "leading dimension too small");
    int64_t g = (rows * n + 255) / 256;
    if (g > kBwdMaxBlocks * 4) g = kBwdMaxBlocks * 4;
    act_bwd_kernel<<<(unsigned)g, 256, 0, (cudaStream_t)stream>>>(Y, ldy, dY, lddy, dX, lddx, rows, n, act);
    return check_launch("lpf_act_backward");
}

extern "C" int lpf_gather_links_backward(const int64_t* links, int64_t bs, const int32_t* idx, int64_t n, const float* X,
                                         int64_t ldx, int32_t d, const float* dsum, int64_t ld_sum, const float* dprod,
                                         int64_t ld_prod, float* dX, int64_t lddx, void* stream) {
    LPF_REQUIRE(bs >= 0 && n >= 0 && d >= 1, "bad shape");
    LPF_REQUIRE(idx || n == bs, "n must equal bs when idx is NULL");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(links && dX && (dsum || dprod), "NULL argument");
    LPF_REQUIRE(!dprod || X, "dprod needs X");
    LPF_REQUIRE((!dsum || ld_sum >= d) && (!dprod || (ld_prod >= d && ldx >= d)) && lddx >= d, "leading dimension too small");
    gather_links_bwd_kernel<<<bwd_grid(n), 256, 0, (cudaStream_t)stream>>>(links, bs, idx, n, X, ldx, d, dsum, ld_sum, dprod,
                                                                          ld_prod, dX, lddx);
    return check_launch("lpf_gather_links_backward");
}

extern "C" int64_t lpf_scatter_rows_backward_workspace_bytes(int64_t rows, int32_t d) {
    if (rows < 0 || d < 1) return -1;
    return ((rows + 15) / 16) * 16 + (int64_t)bwd_grid(rows) * d * (int64_t)sizeof(float);
}

extern "C" int lpf_scatter_rows_backward(const float* dG, int64_t ldg, int64_t rows, int32_t d, const int32_t* idx,
                                         int64_t n, float* dsrc, int64_t ld_src, float* dfill, void* workspace,
                                         int64_t workspace_bytes, void* stream) {
    LPF_REQUIRE(rows >= 0 && n >= 0 && d >= 1 && d <= 4096, "bad shape");
    LPF_REQUIRE(rows == 0 || (dG && ldg >= d), "dG is NULL or ldg < d");
    LPF_REQUIRE(n == 0 || (idx && (!dsrc || ld_src >= d)), "idx is NULL or ld_src < d");
    LPF_REQUIRE(!dfill || (workspace && workspace_bytes >= lpf_scatter_rows_backward_workspace_bytes(rows, d)),
                "workspace too small");
    LPF_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 15) == 0, "workspace must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    uint8_t* mark = dfill ? static_cast<uint8_t*>(workspace) : nullptr;
    float* part = dfill ? reinterpret_cast<float*>(static_cast<char*>(workspace) + ((rows + 15) / 16) * 16) : nullptr;
    if (mark && rows > 0) {
        cudaError_t e = cudaMemsetAsync(mark, 0, (size_t)rows, st);
        if (e != cudaSuccess) { set_error("lpf_scatter_rows_backward: cudaMemsetAsync: %s", cudaGetErrorString(e)); return LPF_ERR_CUDA; }
    }
    if (n > 0 && (dsrc || mark)) {
        int64_t g = (n * d + 255) / 256;
        if (g > kBwdMaxBlocks * 4) g = kBwdMaxBlocks * 4;
        scatter_rows_bwd_gather_kernel<<<(unsigned)g, 256, 0, st>>>(dG, ldg, idx, n, d, dsrc, ld_src, mark);
    }
    if (dfill) {
        const unsigned grid = bwd_grid(rows);
        const size_t smem = (size_t)kBwdWarps * d * sizeof(float);
        cudaError_t e = cudaFuncSetAttribute(masked_colsum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)(kBwdWarps * 4096 * sizeof(float)));
        if (e != cudaSuccess) { set_error("lpf_scatter_rows_backward: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return LPF_ERR_CUDA; }
        masked_colsum_kernel<<<grid, kBwdThreads, smem, st>>>(dG, ldg, rows, d, mark, part);
        launch_reduce(part, grid, d, d, dfill, 0, st);
    }
    return check_launch("lpf_scatter_rows_backward");
}

extern "C" int64_t lpf_rpe_hidden_backward_workspace_bytes(int64_t rows, int32_t d) {
    if (rows < 0 || d < 1) return -1;
    return (int64_t)bwd_grid(rows) * 5 * d * (int64_t)sizeof(float);
}

extern "C" int lpf_rpe_hidden_backward(const float* src_ppr, const float* tgt_ppr, int64_t row0, int64_t rows,
                                       const float* w1, const float* b1, const float* ln_w, const float* ln_b, int32_t d,
                                       const float* dh, int64_t ld_dh, float* dw1, float* db1, float* dln_w, float* dln_b,
                                       int accumulate, void* workspace, int64_t workspace_bytes, void* stream) {
    LPF_REQUIRE(rows >= 0 && row0 >= 0, "negative row range");
    LPF_REQUIRE(d >= 1 && d <= 256, "d must be in [1,256]");
    LPF_REQUIRE(w1 && b1 && ln_w && ln_b && dw1 && db1 && dln_w && dln_b, "NULL argument");
    LPF_REQUIRE(rows == 0 || (src_ppr && tgt_ppr && dh && ld_dh >= d), "NULL pair arrays or ld_dh < d");
    LPF_REQUIRE(workspace && workspace_bytes >= lpf_rpe_hidden_backward_workspace_bytes(rows, d), "workspace too small");
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = bwd_grid(rows);
    float* part = static_cast<float*>(workspace);
    const int kc = (d + 31) / 32;
#define LPF_RPE_BWD(KC) rpe_hidden_bwd_kernel<KC><<<grid, kBwdThreads, 0, st>>>(src_ppr, tgt_ppr, row0, rows, w1, b1, ln_w, ln_b, d, dh, ld_dh, part)
    if (kc <= 1) LPF_RPE_BWD(1);
    else if (kc <= 2) LPF_RPE_BWD(2);
    else if (kc <= 4) LPF_RPE_BWD(4);
    else LPF_RPE_BWD(8);
#undef LPF_RPE_BWD
    rpe_reduce_kernel<<<(unsigned)((5 * d + 255) / 256), 256, 0, st>>>(part, grid, d, dw1, db1, dln_w, dln_b, accumulate);
    return check_launch("lpf_rpe_hidden_backward");
}

extern "C" int lpf_attend_backward(const int64_t* ptr, int64_t bs, const int32_t* idx, int64_t n, const int32_t* node,
                                   const float* KV, int64_t ld_kv, const float* R, int64_t ld_r, const int32_t* r_map,
                                   const float* r_const, const float* Q, int64_t ld_q, const float* att, const float* bias,
                                   const float* ln_w, const float* ln_b, int32_t heads, int32_t ch, const float* dY,
                                   int64_t ld_dy, float* dR, int64_t ld_dr, float* dR_const, float* dQ, int64_t ld_dq,
                                   float* dKV, int64_t ld_dkv, float* link_rows, void* stream) {
    LPF_REQUIRE(bs >= 0 && n >= 0, "negative batch size");
    LPF_REQUIRE(idx || n == bs, "n must equal bs when idx is NULL");
    if (n == 0) return LPF_OK;
    LPF_REQUIRE(ptr && KV && Q && att && bias && ln_w && ln_b && dY && dQ && dKV && link_rows, "NULL argument");
    LPF_REQUIRE(heads >= 1 && ch >= 1, "bad heads/ch");
    const int hc = heads * ch;
    LPF_REQUIRE(ld_kv >= hc && ld_q >= hc && ld_dy >= hc && ld_dq >= hc && ld_dkv >= hc, "leading dimension too small");
    LPF_REQUIRE(R == nullptr || (ld_r >= hc && dR && ld_dr >= hc), "R needs dR (ld_r, ld_dr >= heads*ch)");
    LPF_REQUIRE(r_map == nullptr || (r_const && dR_const), "r_map needs r_const and dR_const");
    // node / R may be NULL only if every set is empty; the kernel never dereferences them then.
    AttendBwdParams p{ptr, bs, idx, n, node, KV, ld_kv, R, ld_r, r_map, r_const, Q, ld_q, att, bias, ln_w, ln_b, dY, ld_dy,
                      dR, ld_dr, dR_const, dQ, ld_dq, dKV, ld_dkv, link_rows, ch};
    cudaStream_t st = (cudaStream_t)stream;
    switch (heads) {
        case 1: return launch_attend_bwd<1>(p, st);
        case 2: return launch_attend_bwd<2>(p, st);
        case 4: return launch_attend_bwd<4>(p, st);
        case 8: return launch_attend_bwd<8>(p, st);
        default:
            set_error("lpf_attend_backward: heads must be 1, 2, 4 or 8 (got %d)", heads);
            return LPF_ERR_UNSUPPORTED;
    }
}
