// K2 — GCN message passing as a vectorised CSR SpMM with the layer's epilogue fused:
//     Y[r,:] = LN2( residual[r,:] + act( LN1( sum_k val[k] * XW[col[k],:] + bias ) ) )
// (every stage after the sum optional).  Replaces GCNConv's torch_sparse.matmul and the LayerNorm / ReLU / residual
// that follow it in GCN.forward, plus — for the last layer — LinkTransformer.gnn_norm (reference
// models/other_models.py:61-76, models/link_transformer.py:126; PyG 2.2.0 gcn_norm semantics are applied when the
// normalised CSR is built, SURVEY App. C).
//
// The work is a gather of 4d-byte feature rows at random node ids: ~0 flop/byte, bound by how many row reads are in
// flight (tools/gather_probe.cu: a B200 serves ~28 G random 256-byte rows/s when enough of them are outstanding).
// One warp per output row; LPR = d/4 lanes hold one feature row as float4 slices, so a warp reads 32/LPR neighbour
// rows per load instruction (two at d = 64: no idle lanes) and keeps four such instructions in flight; the (col, val)
// pairs of up to 32 neighbours come in with one coalesced read each and are broadcast by shuffle; the partial sums of
// the lane groups meet by shuffle at the end, and the row's LayerNorm statistics are reductions over the same lanes:
// the normalised, activated row is written once instead of being written, re-read and re-written by a second launch.
#include "common.cuh"

namespace lpf {

struct SpmmParams {
    const int64_t* rowptr;
    const int32_t* col;
    const float* val;
    int64_t row0, rows;
    const float* XW;
    int64_t ld_xw;
    const float* bias;
    int d;
    // fused epilogue (all optional)
    const float* ln_w;      // LayerNorm 1 (GCN.lns[i])
    const float* ln_b;
    int relu;
    const float* residual;  // rows indexed like Y (absolute row ids)
    int64_t ld_res;
    const float* ln2_w;     // LayerNorm 2 (gnn_norm after the last layer)
    const float* ln2_b;
    float* Y;
    int64_t ldy;
    // dropout after the activation (DROP kernels only; rule in common.cuh): mask row = node id, column = channel
    const uint64_t* seed;
    int site;
    uint64_t thr;
    float scale;
};

// sum over the LPR lanes of a group (LPR a power of two <= 32, groups aligned)
template <int LPR>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// LPR lanes x CH float4 chunks hold one feature row: d <= 4 * LPR * CH, d % 4 == 0 (chunks beyond d are masked).
// DROP: dropout between the activation and the residual (GCN.forward: conv -> LN -> dropout -> ReLU -> + residual;
// dropout and ReLU commute exactly, since relu(m z s) == m relu(z) s for m in {0, 1} and s > 0).
template <int LPR, int CH, bool DROP>
__global__ void __launch_bounds__(256, 4) gcn_spmm_kernel(const __grid_constant__ SpmmParams p) {
    constexpr int GW = 32 / LPR;          // neighbour rows per load instruction
    constexpr int UN = 4;                 // load instructions in flight (8 measured: no faster)
    const int lane = threadIdx.x & 31;
    const int gl = lane % LPR, grp = lane / LPR;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int d = p.d;
    uint64_t seed = 0;
    if constexpr (DROP) seed = *p.seed;
    bool ok[CH];                          // this lane's chunk q lies inside the row
#pragma unroll
    for (int q = 0; q < CH; ++q) ok[q] = 4 * (gl + q * LPR) < d;
    for (int64_t r = warp; r < p.rows; r += nwarps) {
        const int64_t row = p.row0 + r;
        const int64_t k0 = __ldg(p.rowptr + row), k1 = __ldg(p.rowptr + row + 1);
        float4 acc[CH];
#pragma unroll
        for (int q = 0; q < CH; ++q) acc[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int64_t kb = k0; kb < k1; kb += 32) {
            const int cnt = (int)min((int64_t)32, k1 - kb);
            const int32_t my_c = (lane < cnt) ? __ldg(p.col + kb + lane) : 0;
            const float my_v = (lane < cnt) ? __ldg(p.val + kb + lane) : 0.f;
            for (int j0 = 0; j0 < cnt; j0 += GW * UN) {
                float4 t[UN][CH];
                float w[UN];
#pragma unroll
                for (int u = 0; u < UN; ++u) {
                    const int j = j0 + u * GW + grp;                 // this lane group's neighbour of the step
                    const int32_t c = __shfl_sync(kFull, my_c, j & 31);          // (every lane takes part in both shuffles)
                    const float wv = __shfl_sync(kFull, my_v, j & 31);
                    w[u] = j < cnt ? wv : 0.f;
                    const float4* x = reinterpret_cast<const float4*>(p.XW + (int64_t)c * p.ld_xw) + gl;
#pragma unroll
                    for (int q = 0; q < CH; ++q) t[u][q] = (j < cnt && ok[q]) ? __ldg(x + q * LPR) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < UN; ++u)
#pragma unroll
                    for (int q = 0; q < CH; ++q) {
                        acc[q].x = fmaf(w[u], t[u][q].x, acc[q].x);
                        acc[q].y = fmaf(w[u], t[u][q].y, acc[q].y);
                        acc[q].z = fmaf(w[u], t[u][q].z, acc[q].z);
                        acc[q].w = fmaf(w[u], t[u][q].w, acc[q].w);
                    }
            }
        }
        // the lane groups' partial sums meet: every lane ends with the whole row's value of its channels
#pragma unroll
        for (int o = LPR; o < 32; o <<= 1)
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                acc[q].x += __shfl_xor_sync(kFull, acc[q].x, o);
                acc[q].y += __shfl_xor_sync(kFull, acc[q].y, o);
                acc[q].z += __shfl_xor_sync(kFull, acc[q].z, o);
                acc[q].w += __shfl_xor_sync(kFull, acc[q].w, o);
            }
        float v[CH][4];
#pragma unroll
        for (int q = 0; q < CH; ++q) {
            const int ch = 4 * (gl + q * LPR);
            const float4 b = (p.bias && ok[q]) ? __ldg(reinterpret_cast<const float4*>(p.bias + ch)) : make_float4(0.f, 0.f, 0.f, 0.f);
            v[q][0] = acc[q].x + b.x; v[q][1] = acc[q].y + b.y; v[q][2] = acc[q].z + b.z; v[q][3] = acc[q].w + b.w;
        }
        // LayerNorm (two-pass statistics over the row, eps 1e-5) -> ReLU -> + residual -> LayerNorm 2
        auto layer_norm = [&](const float* g, const float* bt) {
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < CH; ++q) s += (v[q][0] + v[q][1]) + (v[q][2] + v[q][3]);
            const float mean = group_sum<LPR>(s) / (float)d;
            float ss = 0.f;
#pragma unroll
            for (int q = 0; q < CH; ++q)
#pragma unroll
                for (int e = 0; e < 4; ++e) ss = ok[q] ? fmaf(v[q][e] - mean, v[q][e] - mean, ss) : ss;
            const float rstd = rsqrtf(group_sum<LPR>(ss) / (float)d + 1e-5f);
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                if (!ok[q]) continue;             // (masked chunks stay 0)
                const int ch = 4 * (gl + q * LPR);
                const float4 g4 = __ldg(reinterpret_cast<const float4*>(g + ch)), b4 = __ldg(reinterpret_cast<const float4*>(bt + ch));
                v[q][0] = fmaf((v[q][0] - mean) * rstd, g4.x, b4.x);
                v[q][1] = fmaf((v[q][1] - mean) * rstd, g4.y, b4.y);
                v[q][2] = fmaf((v[q][2] - mean) * rstd, g4.z, b4.z);
                v[q][3] = fmaf((v[q][3] - mean) * rstd, g4.w, b4.w);
            }
        };
        if (p.ln_w) layer_norm(p.ln_w, p.ln_b);
        if (p.relu) {
#pragma unroll
            for (int q = 0; q < CH; ++q)
#pragma unroll
                for (int e = 0; e < 4; ++e) v[q][e] = fmaxf(v[q][e], 0.f);
        }
        if constexpr (DROP) {
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                if (!ok[q]) continue;
                const uint4 u = dropout_bits(seed, p.site, row, gl + q * LPR);
                v[q][0] = dropout_apply(v[q][0], u.x, p.thr, p.scale);
                v[q][1] = dropout_apply(v[q][1], u.y, p.thr, p.scale);
                v[q][2] = dropout_apply(v[q][2], u.z, p.thr, p.scale);
                v[q][3] = dropout_apply(v[q][3], u.w, p.thr, p.scale);
            }
        }
        if (p.residual) {
#pragma unroll
            for (int q = 0; q < CH; ++q) {
                if (!ok[q]) continue;
                const float4 rr = __ldg(reinterpret_cast<const float4*>(p.residual + row * p.ld_res + 4 * (gl + q * LPR)));
                v[q][0] += rr.x; v[q][1] += rr.y; v[q][2] += rr.z; v[q][3] += rr.w;
            }
        }
        if (p.ln2_w) layer_norm(p.ln2_w, p.ln2_b);
        if (grp == 0) {
#pragma unroll
            for (int q = 0; q < CH; ++q)
                if (ok[q]) *reinterpret_cast<float4*>(p.Y + row * p.ldy + 4 * (gl + q * LPR)) = make_float4(v[q][0], v[q][1], v[q][2], v[q][3]);
        }
    }
}

// Any width / alignment: one warp per row, scalar channels lane + 32 q (no fused epilogue: the caller runs
// lpf_layernorm_act).
__global__ void __launch_bounds__(256) gcn_spmm_scalar_kernel(const __grid_constant__ SpmmParams p) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    constexpr int MAXC = 4;     // d <= 128
    for (int64_t r = warp; r < p.rows; r += nwarps) {
        const int64_t row = p.row0 + r;
        const int64_t k0 = __ldg(p.rowptr + row), k1 = __ldg(p.rowptr + row + 1);
        float acc[MAXC] = {0.f, 0.f, 0.f, 0.f};
        for (int64_t k = k0; k < k1; ++k) {
            const float w = __ldg(p.val + k);
            const float* x = p.XW + (int64_t)__ldg(p.col + k) * p.ld_xw;
#pragma unroll
            for (int q = 0; q < MAXC; ++q)
                if (lane + 32 * q < p.d) acc[q] = fmaf(w, __ldg(x + lane + 32 * q), acc[q]);
        }
#pragma unroll
        for (int q = 0; q < MAXC; ++q)
            if (lane + 32 * q < p.d) p.Y[row * p.ldy + lane + 32 * q] = acc[q] + (p.bias ? __ldg(p.bias + lane + 32 * q) : 0.f);
    }
}

static bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

// widths the vectorised kernel takes: multiples of 4 up to 512
static bool spmm_vec_shape(int d) { return d % 4 == 0 && d >= 4 && d <= 512; }

template <bool DROP>
static int launch_vec(const SpmmParams& p, unsigned blocks, cudaStream_t st) {
    if (p.d <= 16) gcn_spmm_kernel<4, 1, DROP><<<blocks, 256, 0, st>>>(p);
    else if (p.d <= 32) gcn_spmm_kernel<8, 1, DROP><<<blocks, 256, 0, st>>>(p);
    else if (p.d <= 64) gcn_spmm_kernel<16, 1, DROP><<<blocks, 256, 0, st>>>(p);
    else if (p.d <= 128) gcn_spmm_kernel<32, 1, DROP><<<blocks, 256, 0, st>>>(p);
    else if (p.d <= 256) gcn_spmm_kernel<32, 2, DROP><<<blocks, 256, 0, st>>>(p);
    else if (p.d <= 384) gcn_spmm_kernel<32, 3, DROP><<<blocks, 256, 0, st>>>(p);
    else gcn_spmm_kernel<32, 4, DROP><<<blocks, 256, 0, st>>>(p);
    return check_launch("lpf_gcn_spmm");
}

static int launch_spmm(const SpmmParams& p, bool fused_requested, cudaStream_t st) {
    const bool vec = spmm_vec_shape(p.d) && p.ld_xw % 4 == 0 && p.ldy % 4 == 0 && aligned16(p.XW) && aligned16(p.Y) &&
                     (!p.bias || aligned16(p.bias)) && (!p.residual || (aligned16(p.residual) && p.ld_res % 4 == 0)) &&
                     (!p.ln_w || (aligned16(p.ln_w) && aligned16(p.ln_b))) && (!p.ln2_w || (aligned16(p.ln2_w) && aligned16(p.ln2_b)));
    int64_t blocks = (p.rows + 7) / 8;
    const int64_t cap = (int64_t)kNumSMs * 8 * 8;
    if (blocks > cap) blocks = cap;
    if (!vec) {
        if (fused_requested) {
            set_error("lpf_gcn_layer: the fused epilogue needs d %% 4 == 0, d <= 512 and 16-byte aligned rows");
            return LPF_ERR_UNSUPPORTED;
        }
        if (p.d > 128) {
            set_error("lpf_gcn_spmm: d = %d needs 16-byte aligned rows and d %% 4 == 0 (scalar path: d <= 128)", p.d);
            return LPF_ERR_UNSUPPORTED;
        }
        gcn_spmm_scalar_kernel<<<(unsigned)blocks, 256, 0, st>>>(p);
        return check_launch("lpf_gcn_spmm");
    }
    if (p.seed) return launch_vec<true>(p, (unsigned)blocks, st);
    return launch_vec<false>(p, (unsigned)blocks, st);
}

}  // namespace lpf

using namespace lpf;

extern "C" int lpf_gcn_spmm(const int64_t* rowptr, const int32_t* col, const float* val, int64_t row0, int64_t rows,
                            const float* XW, int64_t ld_xw, const float* bias, int32_t d, float* Y, int64_t ldy,
                            void* stream) {
    LPF_REQUIRE(rows >= 0 && row0 >= 0, "negative row range");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(rowptr && XW && Y, "NULL argument");
    LPF_REQUIRE(d >= 1 && ld_xw >= d && ldy >= d, "bad d / leading dimension");
    SpmmParams p{rowptr, col, val, row0, rows, XW, ld_xw, bias, d, nullptr, nullptr, 0, nullptr, 0, nullptr, nullptr, Y, ldy};
    return launch_spmm(p, false, (cudaStream_t)stream);
}

extern "C" int lpf_gcn_layer(const int64_t* rowptr, const int32_t* col, const float* val, int64_t row0, int64_t rows,
                             const float* XW, int64_t ld_xw, const float* bias, int32_t d, const float* ln_w,
                             const float* ln_b, int relu, const float* residual, int64_t ld_res, const float* ln2_w,
                             const float* ln2_b, float* Y, int64_t ldy, void* stream) {
    LPF_REQUIRE(rows >= 0 && row0 >= 0, "negative row range");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(rowptr && XW && Y, "NULL argument");
    LPF_REQUIRE(d >= 1 && ld_xw >= d && ldy >= d && (!residual || ld_res >= d), "bad d / leading dimension");
    LPF_REQUIRE((ln_w == nullptr) == (ln_b == nullptr) && (ln2_w == nullptr) == (ln2_b == nullptr),
                "LayerNorm weight and bias must both be given or both NULL");
    SpmmParams p{rowptr, col, val, row0, rows, XW, ld_xw, bias, d, ln_w, ln_b, relu, residual, ld_res, ln2_w, ln2_b, Y, ldy};
    return launch_spmm(p, true, (cudaStream_t)stream);
}

extern "C" int lpf_gcn_layer_dropout(const int64_t* rowptr, const int32_t* col, const float* val, int64_t row0,
                                     int64_t rows, const float* XW, int64_t ld_xw, const float* bias, int32_t d,
                                     const float* ln_w, const float* ln_b, int relu, const uint64_t* seed, int32_t site,
                                     double p, const float* residual, int64_t ld_res, const float* ln2_w,
                                     const float* ln2_b, float* Y, int64_t ldy, void* stream) {
    LPF_REQUIRE(rows >= 0 && row0 >= 0, "negative row range");
    SpmmParams prm{rowptr, col, val, row0, rows, XW, ld_xw, bias, d, ln_w, ln_b, relu, residual, ld_res, ln2_w, ln2_b, Y, ldy,
                   seed, site, 0, 0.f};
    LPF_REQUIRE(dropout_rule(p, &prm.thr, &prm.scale), "p must be in [0, 1]");
    LPF_REQUIRE(seed, "seed is NULL");
    if (rows == 0) return LPF_OK;
    LPF_REQUIRE(rowptr && XW && Y, "NULL argument");
    LPF_REQUIRE(d >= 1 && ld_xw >= d && ldy >= d && (!residual || ld_res >= d), "bad d / leading dimension");
    LPF_REQUIRE((ln_w == nullptr) == (ln_b == nullptr) && (ln2_w == nullptr) == (ln2_b == nullptr),
                "LayerNorm weight and bias must both be given or both NULL");
    return launch_spmm(prm, true, (cudaStream_t)stream);
}
