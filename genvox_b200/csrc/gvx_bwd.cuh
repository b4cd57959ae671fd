// genvox_b200 — backward through time of the Tacotron2 decoder recurrence.
//
// The reference has no backward source: `loss["loss"].backward()` at
// /root/reference/models/tts/tacotron2.py:520 drives torch autograd over the graph built by
// Decoder.forward (:365-388).  Here the reverse-time chain (what is truly sequential) runs as
// five launches per step; every gradient that is a sum over time (all weight gradients,
// d processed_memory, d memory) is computed afterwards by time-batched GEMMs / reductions:
//   per step t = T-1..0:
//     S1  decoder-LSTM pointwise backward                      -> DGD[t]
//     S2  d x_dec = DGD[t] . W_dec          (skinny GEMM)      -> d h_att, d ctx, d h_dec(t-1)
//     S3  attention backward (gvx_attention.cuh)               -> d e, d q, d conv, d w/d cum carries
//     S4  d h_att += d q . W_query, attention-LSTM pointwise backward (fused epilogue) -> DGA[t]
//     S5  d x_att = DGA[t] . W_att          (skinny GEMM)      -> d prenet_out, d ctx(t-1), d h_att(t-1)
//   afterwards: cuBLAS sgemm (plain time-batched GEMMs) for d W of both LSTMs, projection, query,
//   memory layer, prenet; custom reductions for d v / d location_dense / d location_conv / d pm.
#pragma once
#include <cublas_v2.h>

#include "../../include/genvox_b200.h"
#include "gvx_attention_c2.cuh"
#include "gvx_blas.cuh"
#include "gvx_common.cuh"
#include "gvx_gemm.cuh"
#include "gvx_layout.cuh"
#include "gvx_misc.cuh"
#include "gvx_post_tc.cuh"

namespace gvx {

// S1: decoder-LSTM pointwise backward.  d h_dropped = dh1 (+ dh2)
__global__ void k_lstm_bwd_pointwise(const float *__restrict__ dh1, int ld1, const float *__restrict__ dh2, int ld2,
                                     DropCfg drop, uint32_t site, uint32_t t, int row_offset,
                                     const float *__restrict__ gates, const float *__restrict__ c_prev,
                                     const float *__restrict__ c_new, float *__restrict__ dc, float *__restrict__ dgates,
                                     int B, int HID) {
    pdl_trigger();
    pdl_wait();
    const int total = B * HID;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int b = i / HID, u = i - b * HID;
        float dh = dh1[(size_t)b * ld1 + u];
        if (dh2) dh += dh2[(size_t)b * ld2 + u];
        const float mult = drop_mult(drop, site, t, (uint32_t)(b + row_offset), (uint32_t)u);
        const float4 ga = *reinterpret_cast<const float4 *>(gates + (size_t)b * 4 * HID + 4 * u);
        float dcp;
        const float4 dp = lstm_bwd_point(dh, mult, ga, c_prev[i], c_new[i], dc[i], dcp);
        dc[i] = dcp;
        *reinterpret_cast<float4 *>(dgates + (size_t)b * 4 * HID + 4 * u) = dp;
    }
}

// prenet backward mask: dz = dy * 2 * [y > 0]   (y = relu(z) * keep * 2, tacotron2.py:143)
__global__ void k_prenet_bwd_mask(const float *dy, int ldy, const float *__restrict__ y, int rows, int P, float *dz) {
    const size_t total = (size_t)rows * P;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / P;
        const int c = (int)(i - r * P);
        dz[i] = y[i] > 0.f ? 2.f * dy[r * ldy + c] : 0.f;
    }
}

// packed bias gradient [4*HID] (row 4u+g) -> torch order (g*HID+u), written to both b_ih and b_hh
__global__ void k_unpack_bias_grad(const float *__restrict__ db, int HID, float *__restrict__ d_ih, float *__restrict__ d_hh) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 4 * HID; i += gridDim.x * blockDim.x) {
        const int u = i >> 2, g = i & 3;
        d_ih[g * HID + u] = db[i];
        d_hh[g * HID + u] = db[i];
    }
}

// Post-pass 1: for every token (b, n), over all t:  d s = d e * v * (1 - th^2)
//   d pm[b,n,d] = sum_t d s;  d v[d] += sum d e * th;  d Wld[d,f] += sum d s * conv[f]
// blockDim = D threads (thread = d), 8 resident blocks per SM and a 4-deep unrolled time loop keep enough
// loads in flight to stream the [T,B,N,D] tanh stash near HBM speed; per-block partials of d Wld / d v are
// reduced in a fixed order by k_reduce_partials.
template <int FMAX>
__global__ void __launch_bounds__(512, (FMAX <= 32 ? 2 : 1)) k_attn_post_dense(const float *__restrict__ TH, const float *__restrict__ DE,
                                                             const float *__restrict__ CONVS, const float *__restrict__ v, int T,
                                                             int B, int N, int D, int F, float *__restrict__ DPM,
                                                             float *__restrict__ part /* [grid][D*F + D] */) {
    const int d = threadIdx.x;
    float wacc[FMAX];
#pragma unroll
    for (int f = 0; f < FMAX; ++f) wacc[f] = 0.f;
    float vacc = 0.f;
    const float vd = d < D ? v[d] : 0.f;
    const size_t tok_stride = (size_t)B * N;
    for (int tok = blockIdx.x; tok < B * N; tok += gridDim.x) {
        float pacc = 0.f;
        int t = 0;
        for (; t + 4 <= T; t += 4) {
            float de[4], th[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const size_t row = (size_t)(t + i) * tok_stride + tok;
                de[i] = DE[row];
                th[i] = d < D ? TH[row * D + d] : 0.f;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const size_t row = (size_t)(t + i) * tok_stride + tok;
                const float ds = de[i] * vd * (1.f - th[i] * th[i]);
                pacc += ds;
                vacc = fmaf(de[i], th[i], vacc);
                const float4 *cv = reinterpret_cast<const float4 *>(CONVS + row * F);
                if (FMAX % 4 == 0 && F == FMAX) {
#pragma unroll
                    for (int f4 = 0; f4 < FMAX / 4; ++f4) {
                        const float4 c = cv[f4];
                        wacc[4 * f4] = fmaf(ds, c.x, wacc[4 * f4]); wacc[4 * f4 + 1] = fmaf(ds, c.y, wacc[4 * f4 + 1]);
                        wacc[4 * f4 + 2] = fmaf(ds, c.z, wacc[4 * f4 + 2]); wacc[4 * f4 + 3] = fmaf(ds, c.w, wacc[4 * f4 + 3]);
                    }
                } else {
                    const float *cs = CONVS + row * F;
#pragma unroll
                    for (int f = 0; f < FMAX; ++f)
                        if (f < F) wacc[f] = fmaf(ds, cs[f], wacc[f]);
                }
            }
        }
        for (; t < T; ++t) {
            const size_t row = (size_t)t * tok_stride + tok;
            const float de = DE[row];
            const float th = d < D ? TH[row * D + d] : 0.f;
            const float ds = de * vd * (1.f - th * th);
            pacc += ds;
            vacc = fmaf(de, th, vacc);
            const float *cs = CONVS + row * F;
#pragma unroll
            for (int f = 0; f < FMAX; ++f)
                if (f < F) wacc[f] = fmaf(ds, cs[f], wacc[f]);
        }
        if (d < D) DPM[(size_t)tok * D + d] = pacc;
    }
    if (d < D) {
        float *p = part + (size_t)blockIdx.x * (D * F + D);
#pragma unroll
        for (int f = 0; f < FMAX; ++f)
            if (f < F) p[d * F + f] = wacc[f];
        p[D * F + d] = vacc;
    }
}


// Post-pass 1 on tensor cores (bf16 mode, att_dim 128 / 32 location filters).  The FFMA kernel above issues ~47
// instructions per (token, frame, d) and reaches ~0.9 TB/s of the 5 GB it streams (ncu, T = 800: 5.4 ms); the outer
// product  d Wld[d, f] += sum_t d s[t, d] * conv[t, f]  is a [128 x 16] . [16 x 32] contraction per 16 frames of a token:
//   thread = attention dim d: loads th[t0..t0+15][d] (16 independent coalesced loads), forms d s, keeps the d pm / d v
//   sums in fp32, packs frame pairs to bf16x2 and stores them as the A operand ([d][t], padded rows: conflict-free
//   fragment reads); the conv rows of the chunk become the B operand ([f][t]) the same way;
//   warp w contracts d rows [32w, 32w+32) x all 32 filters: 8 mma.sync.m16n8k16 per chunk, fp32 accumulators.
// Operands are rounded to bf16 (as in every contraction of bf16 mode); accumulation and the d pm / d v sums stay fp32.
constexpr int PDM_TC = 16;         // frames per chunk = one MMA k-step
constexpr int PDM_LDA = 12;        // 32-bit words per operand row (8 used): bank = 12 g + tig is conflict-free
__device__ __forceinline__ void pdm_mma(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pdm_pack(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t *>(&v);
}
template <bool THBF>     // THBF: the tanh stash is bf16 with 16-byte chunks swizzled by (token & 7) (written by k_att_chain_fwd)
__global__ void __launch_bounds__(128, 5) k_attn_post_dense_mma(const float *__restrict__ TH, const float *__restrict__ DE,
                                                                const float *__restrict__ CONVS, const float *__restrict__ v, int T,
                                                                int B, int N, float *__restrict__ DPM,
                                                                float *__restrict__ part /* [grid][128*32 + 128] */) {
    constexpr int D = 128, F = 32;
    __shared__ __align__(16) uint32_t sA[2][D * PDM_LDA];      // [d][frame pair] bf16x2
    __shared__ __align__(16) uint32_t sB[2][F * PDM_LDA];      // [f][frame pair] bf16x2
    const int d = threadIdx.x, warp = d >> 5, lane = d & 31, g = lane >> 2, tig = lane & 3;
    const float vd = v[d];
    const size_t tok_stride = (size_t)B * N;
    float acc[2][4][4];                                        // [m-tile][n-tile][fragment]
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[m][n][i] = 0.f;
    float vacc = 0.f;
    // conv staging: thread -> (frame pair p, filter pair q): conv[2p..2p+1][2q..2q+1]
    const int cp_ = d >> 4, cq = d & 15;
    int buf = 0;
    const unsigned short *THB = reinterpret_cast<const unsigned short *>(TH);
    for (int tok = blockIdx.x; tok < B * N; tok += gridDim.x) {
        float pacc = 0.f;
        const int dsw = ((((d >> 3) ^ ((tok % N) & 7)) << 3) | (d & 7));
        for (int t0 = 0; t0 < T; t0 += PDM_TC) {
            float th[PDM_TC], de[PDM_TC];
#pragma unroll
            for (int i = 0; i < PDM_TC; ++i) {
                const bool in = t0 + i < T;
                const size_t row = (size_t)(in ? t0 + i : 0) * tok_stride + tok;
                if (THBF) th[i] = in ? __uint_as_float((unsigned)__ldcs(THB + row * D + dsw) << 16) : 0.f;
                else th[i] = in ? __ldcs(TH + row * D + d) : 0.f;
                de[i] = in ? __ldg(DE + row) : 0.f;
            }
            float2 c0 = make_float2(0.f, 0.f), c1 = make_float2(0.f, 0.f);
            {
                const int ta = t0 + 2 * cp_;
                if (ta < T) c0 = __ldcs(reinterpret_cast<const float2 *>(CONVS + ((size_t)ta * tok_stride + tok) * F + 2 * cq));
                if (ta + 1 < T) c1 = __ldcs(reinterpret_cast<const float2 *>(CONVS + ((size_t)(ta + 1) * tok_stride + tok) * F + 2 * cq));
            }
            uint32_t pk[PDM_TC / 2];
#pragma unroll
            for (int i = 0; i < PDM_TC; i += 2) {
                const float ds0 = de[i] * vd * (1.f - th[i] * th[i]), ds1 = de[i + 1] * vd * (1.f - th[i + 1] * th[i + 1]);
                pacc += ds0 + ds1;
                vacc = fmaf(de[i], th[i], vacc);
                vacc = fmaf(de[i + 1], th[i + 1], vacc);
                pk[i / 2] = pdm_pack(ds0, ds1);
            }
            uint4 *arow = reinterpret_cast<uint4 *>(&sA[buf][d * PDM_LDA]);
            arow[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
            arow[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
            sB[buf][(2 * cq) * PDM_LDA + cp_] = pdm_pack(c0.x, c1.x);
            sB[buf][(2 * cq + 1) * PDM_LDA + cp_] = pdm_pack(c0.y, c1.y);
            __syncthreads();          // the other buffer is free again once every warp has passed this barrier twice
            uint32_t bfr[4][2];
#pragma unroll
            for (int n = 0; n < 4; ++n) {
                bfr[n][0] = sB[buf][(8 * n + g) * PDM_LDA + tig];
                bfr[n][1] = sB[buf][(8 * n + g) * PDM_LDA + tig + 4];
            }
#pragma unroll
            for (int m = 0; m < 2; ++m) {
                const int r0 = 32 * warp + 16 * m + g;
                const uint32_t a0 = sA[buf][r0 * PDM_LDA + tig], a1 = sA[buf][(r0 + 8) * PDM_LDA + tig];
                const uint32_t a2 = sA[buf][r0 * PDM_LDA + tig + 4], a3 = sA[buf][(r0 + 8) * PDM_LDA + tig + 4];
#pragma unroll
                for (int n = 0; n < 4; ++n) pdm_mma(acc[m][n], a0, a1, a2, a3, bfr[n][0], bfr[n][1]);
            }
            buf ^= 1;
        }
        DPM[(size_t)tok * D + d] = pacc;
    }
    float *p = part + (size_t)blockIdx.x * (D * F + D);
#pragma unroll
    for (int m = 0; m < 2; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) {
            const int r0 = 32 * warp + 16 * m + g, c0 = 8 * n + 2 * tig;
            p[r0 * F + c0] = acc[m][n][0];
            p[r0 * F + c0 + 1] = acc[m][n][1];
            p[(r0 + 8) * F + c0] = acc[m][n][2];
            p[(r0 + 8) * F + c0 + 1] = acc[m][n][3];
        }
    p[D * F + d] = vacc;
}

// Post-pass 2: d Wlc[f,c,k] = sum_{t,b,n} d conv[t,b,n,f] * wcat[t,b,c,n+k-pad]
//   wcat channel 0 = alignments of step t-1 (zeros at t = 0), channel 1 = cum before step t.
// One thread = (filter f, channel c, block of 8 taps); the 8-tap window slides over the tokens in registers
// (6 LDS.128 per 64 FMAs).  Per-block partials [grid][F*2*KS], reduced afterwards in a fixed order.
__global__ void __launch_bounds__(1024, 1) k_attn_post_conv(const float *__restrict__ DCONV, const float *__restrict__ ALIGN,
                                                              const float *__restrict__ CUMS, int T, int B, int N, int F, int KS,
                                                              float *__restrict__ part /* [grid][F*2*KS] */) {
    extern __shared__ __align__(16) float sm[];
    const int pad = (KS - 1) / 2, KB = (KS + 7) / 8;
    const int NCS = (N + 7) & ~7, NPS = NCS + 8 * KB + 8;
    float *wc = sm;                         // [2][NPS], index = token + pad
    float *dT = sm + 2 * NPS;               // [F][NCS]
    const int ntask = F * 2 * KB;
    const int task = threadIdx.x;
    const int f = task / (2 * KB), c = (task / KB) & 1, k0 = (task % KB) * 8;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int item = blockIdx.x; item < T * B; item += gridDim.x) {
        const int t = item / B, b = item - t * B;
        __syncthreads();
        for (int i = threadIdx.x; i < 2 * NPS; i += blockDim.x) {
            const int cc = i / NPS, n = i - cc * NPS - pad;
            float x = 0.f;
            if (n >= 0 && n < N) {
                if (cc == 0) x = t > 0 ? ALIGN[((size_t)b * T + (t - 1)) * N + n] : 0.f;
                else x = CUMS[((size_t)b * T + t) * N + n];
            }
            wc[i] = x;
        }
        const float *src = DCONV + ((size_t)t * B + b) * N * F;
        for (int i = threadIdx.x; i < NCS * F; i += blockDim.x) {
            const int n = i / F, ff = i - n * F;
            dT[ff * NCS + n] = n < N ? src[i] : 0.f;
        }
        __syncthreads();
        if (task < ntask) {
            const float *dr = dT + f * NCS, *xr = wc + c * NPS + k0;
            for (int n0 = 0; n0 < NCS; n0 += 8) {
                const float4 d0 = *reinterpret_cast<const float4 *>(dr + n0), d1 = *reinterpret_cast<const float4 *>(dr + n0 + 4);
                const float dd[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
                float x[16];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float4 t4 = *reinterpret_cast<const float4 *>(xr + n0 + 4 * i);
                    x[4 * i] = t4.x; x[4 * i + 1] = t4.y; x[4 * i + 2] = t4.z; x[4 * i + 3] = t4.w;
                }
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[j] = fmaf(dd[i], x[i + j], acc[j]);
            }
        }
    }
    if (task < ntask) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (k0 + j < KS) part[(size_t)blockIdx.x * (F * 2 * KS) + (f * 2 + c) * KS + k0 + j] = acc[j];
    }
}

// out[i] = sum_blk part[blk * stride + off + i]: 8 interleaved groups of blocks per output (threadIdx.y), each
// summed in order, then combined in a fixed order -> deterministic, 8x more loads in flight than a single loop
__global__ void __launch_bounds__(256) k_reduce_partials(const float *__restrict__ part, int nblk, int stride, int off, int n,
                                                          float *__restrict__ out) {
    __shared__ float sh[8][32];
    const int i = blockIdx.x * 32 + threadIdx.x, g = threadIdx.y;
    float s = 0.f;
    if (i < n)
        for (int k = g; k < nblk; k += 8) s += part[(size_t)k * stride + off + i];
    sh[g][threadIdx.x] = s;
    __syncthreads();
    if (g == 0 && i < n) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) t += sh[q][threadIdx.x];
        out[i] = t;
    }
}

// Everything after the reverse-time chain that does not depend on the precision mode:
// attention parameters (sums over t, b, n), memory layer, d memory, prenet.  DZ2 must already hold
// d z2 = 2 [PRE2 > 0] d PRE2.
struct BwdPostArgs {
    const float *TH, *DE, *CONVS, *DCONV, *ALIGN, *CUMS, *DCTX, *PRE1, *FR;
    float *DPM, *PART1, *PART2, *DZ2, *DZ1;
    int post_blocks;
    int bf16_mode;            // 1: bf16-operand tensor-core post-pass for d location_dense (gvx_bf16_api.cuh), 0: exact fp32
    int th_bf16 = 0;          // the tanh stash is bf16 / chunk-swizzled (fused persistent chains)
};
inline int bwd_post_common(const Dims &d, const gvx_weights *w, const float *memory, int B, int N, int T, const BwdPostArgs &p,
                           const gvx_grads *g, float *d_memory, cudaStream_t st) {
    const int TB = T * B;
    {
        const int nblk = p.post_blocks;
        const int threads = (d.D + 31) & ~31;
        GVX_CHECK(threads <= 512, "att_dim too large");
        const bool stream = p.th_bf16 && p.bf16_mode && d.D == 128 && d.F == 32 && d.KS == 31;
        int nblk1 = nblk, nblk2 = nblk;
        if (stream) {
            // fused persistent chains: bf16 tanh stash (chunk-swizzled) and bf16 d conv rows -> the streaming kernels of gvx_post_tc.cuh
            const int items = B * ((N + PT_TOK - 1) / PT_TOK);
            nblk1 = items < nblk ? items : nblk;
            k_post_dense_stream<<<nblk1, 128, 0, st>>>(reinterpret_cast<const uint16_t *>(p.TH), p.DE, p.CONVS, w->v_w, T, B, N, p.DPM, p.PART1);
        } else if (p.bf16_mode && d.D == 128 && d.F == 32) {
            k_attn_post_dense_mma<false><<<nblk, 128, 0, st>>>(p.TH, p.DE, p.CONVS, w->v_w, T, B, N, p.DPM, p.PART1);
        } else if (d.F <= 32) {
            k_attn_post_dense<32><<<nblk, threads, 0, st>>>(p.TH, p.DE, p.CONVS, w->v_w, T, B, N, d.D, d.F, p.DPM, p.PART1);
        } else {
            k_attn_post_dense<64><<<nblk, threads, 0, st>>>(p.TH, p.DE, p.CONVS, w->v_w, T, B, N, d.D, d.F, p.DPM, p.PART1);
        }
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
        const int stride = d.D * d.F + d.D;
        k_reduce_partials<<<(d.D * d.F + 31) / 32, dim3(32, 8), 0, st>>>(p.PART1, nblk1, stride, 0, d.D * d.F, g->loc_dense_w);
        GVX_LAUNCHED(1);
        k_reduce_partials<<<(d.D + 31) / 32, dim3(32, 8), 0, st>>>(p.PART1, nblk1, stride, d.D * d.F, d.D, g->v_w);
        GVX_LAUNCHED(1);
        if (stream) {
            const PtConvGeom cg(N);
            const size_t smem = (size_t)PT_CSTAGES * cg.stage_bytes;
            GVX_CHECK(smem <= 200 * 1024, "token count too large for the conv-gradient kernel");
            static size_t configured = 0;
            if (smem > configured) {
                GVX_CUDA(cudaFuncSetAttribute(k_post_conv_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                configured = smem;
            }
            nblk2 = T * B < nblk / 2 ? T * B : nblk / 2;
            k_post_conv_stream<<<nblk2, 128, smem, st>>>(reinterpret_cast<const uint16_t *>(p.DCONV), p.ALIGN, p.CUMS, T, B, N, p.PART2);
        } else {
            const int KB = (d.KS + 7) / 8, NCS = (N + 7) & ~7, NPS = NCS + 8 * KB + 8;
            const int cthreads = (d.F * 2 * KB + 31) & ~31;
            GVX_CHECK(cthreads <= 1024, "location conv too large for the conv-gradient kernel");
            const size_t smem = ((size_t)2 * NPS + (size_t)d.F * NCS) * sizeof(float);
            GVX_CHECK(smem <= 200 * 1024, "token count too large for the conv-gradient kernel");
            static size_t configured = 0;
            if (smem > configured) {
                GVX_CUDA(cudaFuncSetAttribute(k_attn_post_conv, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                configured = smem;
            }
            k_attn_post_conv<<<nblk, cthreads < 64 ? 64 : cthreads, smem, st>>>(p.DCONV, p.ALIGN, p.CUMS, T, B, N, d.F, d.KS, p.PART2);
        }
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
        k_reduce_partials<<<(d.F * 2 * d.KS + 31) / 32, dim3(32, 8), 0, st>>>(p.PART2, nblk2, d.F * 2 * d.KS, 0, d.F * 2 * d.KS,
                                                                           g->loc_conv_w);
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
    }
    // memory layer and d memory:  d Wm = DPM^T . memory;  d memory = DPM . Wm + align^T . d ctx (per row)
    GVX_TRY(gemm_tn(st, d.D, d.E, B * N, p.DPM, d.D, memory, d.E, g->memory_w, d.E, 0.f));
    GVX_TRY(gemm_nn(st, B * N, d.E, d.D, p.DPM, d.D, w->memory_w, d.E, d_memory, d.E, 0.f));
    {
        cublasHandle_t h;
        GVX_TRY(blas(&h, st));
        const float alpha = 1.f, beta = 1.f;
        // row-major per b: C[N, E] += A[T, N]^T . Bm[T, E];  A = ALIGN[b] (lda N), Bm = DCTX[:, b, :] (ldb B*E)
        GVX_CUBLAS(cublasSgemmStridedBatched(h, CUBLAS_OP_N, CUBLAS_OP_T, d.E, N, T, &alpha, p.DCTX, B * d.E, (long long)d.E,
                                             p.ALIGN, N, (long long)T * N, &beta, d_memory, d.E, (long long)N * d.E, B));
    }
    // prenet (tacotron2.py:140-144): d W1 = d z2^T . PRE1;  d PRE1 = d z2 . W1;  d z1 = 2 [PRE1 > 0] d PRE1;  d W0 = d z1^T . frames
    GVX_TRY(gemm_tn(st, d.P, d.P, TB, p.DZ2, d.P, p.PRE1, d.P, g->prenet_w1, d.P, 0.f));
    GVX_TRY(gemm_nn(st, TB, d.P, d.P, p.DZ2, d.P, w->prenet_w1, d.P, p.DZ1, d.P, 0.f));
    k_prenet_bwd_mask<<<grid_for((size_t)TB * d.P), 256, 0, st>>>(p.DZ1, d.P, p.PRE1, TB, d.P, p.DZ1);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_TRY(gemm_tn(st, d.P, d.M, TB, p.DZ1, d.P, p.FR, d.M, g->prenet_w0, d.M, 0.f));
    return 0;
}

// BPTT in fp32 mode: reads the stash S of train_fwd_fp32, works in W
int train_bwd_fp32(const Dims &d, const StashL &S, const BwdL &W, const gvx_weights *w, const float *packed, const float *memory,
                   const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training, int row_offset, const float *d_mel,
                   const float *d_gate, const float *d_align, const float *s, float *x, const gvx_grads *g, float *d_memory,
                   cudaStream_t st) {
    GVX_CHECK(d.F * 2 * d.KS <= 8 * 512, "location conv too large for the backward reduction kernel");
    const PackedL PL(d);
    const int TB = T * B;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H, BE = (size_t)B * d.E;

    GVX_CUDA(cudaMemsetAsync(x + W.DW, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCUM, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCA, 0, BA * sizeof(float), st));
    k_fill_f32<<<grid_for((size_t)TB), 256, 0, st>>>(x + W.ONES, (size_t)TB, 1.f);
    GVX_LAUNCHED(1);

    // upstream gradients, time-major; d [h_dec | ctx] through the projections for every frame at once
    k_pack_dout<<<grid_for((size_t)TB * d.OL), 256, 0, st>>>(d_mel, d_gate, B, d.M, d.OL, T, x + W.DOUT);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_TRY(gemm_nn(st, TB, d.Kp, d.M + 1, x + W.DOUT, d.OL, packed + PL.Wpg, d.Kp, x + W.DHC, d.Kp, 0.f));

    const DropCfg drop_dec = make_drop(seed, d.p_dec, training), drop_att = make_drop(seed, d.p_att, training);
    pdl_barrier_next();
    for (int t = T - 1; t >= 0; --t) {
        const bool last = t == T - 1;
        float *dxd = x + W.DXD + (size_t)(t & 1) * B * d.Kd;
        const float *dxd_next = x + W.DXD + (size_t)((t + 1) & 1) * B * d.Kd;
        float *dxa = x + W.DXA + (size_t)t * B * d.Ka;
        const float *dxa_next = x + W.DXA + (size_t)(t + 1) * B * d.Ka;
        // S1
        {
        ProfScope ps(PS_BWD_DEC_POINT, st);
        GVX_CUDA(launch_pdl(k_lstm_bwd_pointwise, dim3(grid_for(BH)), dim3(256), 0, st,
            x + W.DHC + (size_t)t * B * d.Kp, d.Kp, last ? nullptr : dxd_next + d.A + d.E, d.Kd, drop_dec, SITE_DEC,
            (uint32_t)t, row_offset, s + S.GD + (size_t)t * 4 * BH, s + S.CD + t * BH, s + S.CD + (t + 1) * BH, x + W.DCD,
            x + W.DGD + (size_t)t * 4 * BH, B, d.H));
        GVX_LAUNCHED(1);
        }
        GVX_CUDA(cudaGetLastError());
        // S2
        {
            ProfScope ps(PS_BWD_DEC_GEMM, st);
            GemmIn gi = gemm_in(packed + PL.WdT, 4 * d.H, d.Kd, B);
            add_seg(gi, x + W.DGD + (size_t)t * 4 * BH, 4 * d.H, 4 * d.H);
            EpiStore e;
            memset(&e, 0, sizeof(e));
            e.out = dxd;
            e.ldo = d.Kd;
            GVX_TRY((launch_gemm<16, EpiStore>(gi, e, st)));
        }
        // S3
        {
            ProfScope ps(PS_BWD_ATTENTION, st);
            AttnBwdArgs a;
            memset(&a, 0, sizeof(a));
            a.s = AttnShape{B, N, d.D, d.E, d.F, d.KS};
            a.memory = memory; a.wlc = w->loc_conv_w; a.wld = w->loc_dense_w; a.v = w->v_w; a.lengths = mem_lengths;
            a.w_t = s + S.ALIGN + (size_t)t * N; a.w_bstride = (long long)T * N;
            a.th = s + S.TH + (size_t)t * B * N * d.D;
            a.dctx1 = src_plain(x + W.DHC + (size_t)t * B * d.Kp + d.H, d.Kp);
            a.dctx2 = src_plain(dxd + d.A, d.Kd);
            a.dctx3 = last ? src_none() : src_plain(dxa_next + d.P, d.Ka);
            a.d_align = d_align ? d_align + (size_t)t * N : nullptr; a.da_bstride = (long long)T * N;
            a.dw_carry = x + W.DW; a.dcum_carry = x + W.DCUM;
            a.dctx_out = x + W.DCTX + t * BE;
            a.de_out = x + W.DE + (size_t)t * B * N;
            a.dq_out = x + W.DQ + (size_t)t * B * d.D;
            a.dconv_out = x + W.DCONV + (size_t)t * B * N * d.F;
            GVX_TRY(launch_attention_bwd_best(a, st));
        }
        // S4
        {
            ProfScope ps(PS_BWD_ATT_POINT, st);
            GemmIn gi = gemm_in(packed + PL.WqT, d.D, d.A, B);
            add_seg(gi, x + W.DQ + (size_t)t * B * d.D, d.D, d.D);
            EpiLstmBwd e;
            memset(&e, 0, sizeof(e));
            e.add1 = dxd; e.ld1 = d.Kd;
            e.add2 = last ? nullptr : dxa_next + d.P + d.E; e.ld2 = d.Ka;
            e.drop = drop_att; e.site = SITE_ATT; e.t = (uint32_t)t; e.row_offset = row_offset;
            e.gates = s + S.GA + (size_t)t * 4 * BA; e.c_prev = s + S.CA + t * BA; e.c_new = s + S.CA + (t + 1) * BA;
            e.dc = x + W.DCA; e.dgates = x + W.DGA + (size_t)t * 4 * BA; e.HID = d.A;
            GVX_TRY((launch_gemm<8, EpiLstmBwd>(gi, e, st)));
        }
        // S5
        {
            ProfScope ps(PS_BWD_ATT_GEMM, st);
            GemmIn gi = gemm_in(packed + PL.WaT, 4 * d.A, d.Ka, B);
            add_seg(gi, x + W.DGA + (size_t)t * 4 * BA, 4 * d.A, 4 * d.A);
            EpiStore e;
            memset(&e, 0, sizeof(e));
            e.out = dxa;
            e.ldo = d.Ka;
            GVX_TRY((launch_gemm<16, EpiStore>(gi, e, st)));
        }
    }

    // ---------------- time-batched gradients ----------------
    ProfScope ps_batched(PS_BWD_BATCHED, st);
    // projections (linear_projection + gate_layer): d Wpg = DOUT^T . [HD[1:], CTX[1:]]
    float *tmp = x + W.TMP;
    GVX_TRY(gemm_tn(st, d.M + 1, d.H, TB, x + W.DOUT, d.OL, s + S.HD + BH, d.H, tmp, d.Kp, 0.f));
    GVX_TRY(gemm_tn(st, d.M + 1, d.E, TB, x + W.DOUT, d.OL, s + S.CTX + BE, d.E, tmp + d.H, d.Kp, 0.f));
    GVX_CUDA(cudaMemcpyAsync(g->proj_w, tmp, (size_t)d.M * d.Kp * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_CUDA(cudaMemcpyAsync(g->gate_w, tmp + (size_t)d.M * d.Kp, (size_t)d.Kp * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_TRY(colsum(st, x + W.DOUT, TB, d.M + 1, d.OL, x + W.ONES, x + W.DBIAS));
    GVX_CUDA(cudaMemcpyAsync(g->proj_b, x + W.DBIAS, (size_t)d.M * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_CUDA(cudaMemcpyAsync(g->gate_b, x + W.DBIAS + d.M, sizeof(float), cudaMemcpyDeviceToDevice, st));

    // decoder LSTM: d Wd (packed) = DGD^T . [HA[1:], CTX[1:], HD[:T]]
    GVX_TRY(gemm_tn(st, 4 * d.H, d.A, TB, x + W.DGD, 4 * d.H, s + S.HA + BA, d.A, x + W.DWD, d.Kd, 0.f));
    GVX_TRY(gemm_tn(st, 4 * d.H, d.E, TB, x + W.DGD, 4 * d.H, s + S.CTX + BE, d.E, x + W.DWD + d.A, d.Kd, 0.f));
    GVX_TRY(gemm_tn(st, 4 * d.H, d.H, TB, x + W.DGD, 4 * d.H, s + S.HD, d.H, x + W.DWD + d.A + d.E, d.Kd, 0.f));
    k_unpack_lstm_grad<<<grid_for((size_t)4 * d.H * d.Kd), 256, 0, st>>>(x + W.DWD, d.H, d.A + d.E, g->dec_w_ih, g->dec_w_hh);
    GVX_LAUNCHED(1);
    GVX_TRY(colsum(st, x + W.DGD, TB, 4 * d.H, 4 * d.H, x + W.ONES, x + W.DBIAS));
    k_unpack_bias_grad<<<grid_for((size_t)4 * d.H), 256, 0, st>>>(x + W.DBIAS, d.H, g->dec_b_ih, g->dec_b_hh);
    GVX_LAUNCHED(1);
    // attention LSTM: d Wa (packed) = DGA^T . [PRE2, CTX[:T], HA[:T]]
    GVX_TRY(gemm_tn(st, 4 * d.A, d.P, TB, x + W.DGA, 4 * d.A, s + S.PRE2, d.P, x + W.DWA, d.Ka, 0.f));
    GVX_TRY(gemm_tn(st, 4 * d.A, d.E, TB, x + W.DGA, 4 * d.A, s + S.CTX, d.E, x + W.DWA + d.P, d.Ka, 0.f));
    GVX_TRY(gemm_tn(st, 4 * d.A, d.A, TB, x + W.DGA, 4 * d.A, s + S.HA, d.A, x + W.DWA + d.P + d.E, d.Ka, 0.f));
    k_unpack_lstm_grad<<<grid_for((size_t)4 * d.A * d.Ka), 256, 0, st>>>(x + W.DWA, d.A, d.P + d.E, g->att_w_ih, g->att_w_hh);
    GVX_LAUNCHED(1);
    GVX_TRY(colsum(st, x + W.DGA, TB, 4 * d.A, 4 * d.A, x + W.ONES, x + W.DBIAS));
    k_unpack_bias_grad<<<grid_for((size_t)4 * d.A), 256, 0, st>>>(x + W.DBIAS, d.A, g->att_b_ih, g->att_b_hh);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    // query layer: d Wq [D, A] = DQ^T . HA[1:]
    GVX_TRY(gemm_tn(st, d.D, d.A, TB, x + W.DQ, d.D, s + S.HA + BA, d.A, g->query_w, d.A, 0.f));

    // prenet mask, then everything that does not depend on the precision mode
    k_prenet_bwd_mask<<<grid_for((size_t)TB * d.P), 256, 0, st>>>(x + W.DXA, d.Ka, s + S.PRE2, TB, d.P, x + W.DZ2);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    BwdPostArgs pa;
    pa.TH = s + S.TH; pa.DE = x + W.DE; pa.CONVS = s + S.CONVS; pa.DCONV = x + W.DCONV; pa.ALIGN = s + S.ALIGN;
    pa.CUMS = s + S.CUMS; pa.DCTX = x + W.DCTX; pa.PRE1 = s + S.PRE1; pa.FR = s + S.FR;
    pa.DPM = x + W.DPM; pa.PART1 = x + W.PART1; pa.PART2 = x + W.PART2; pa.DZ2 = x + W.DZ2; pa.DZ1 = x + W.DZ1;
    pa.post_blocks = W.post_blocks;
    pa.bf16_mode = 0;
    return bwd_post_common(d, w, memory, B, N, T, pa, g, d_memory, st);
}

}  // namespace gvx
