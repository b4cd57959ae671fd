// genvox_b200 — fp32 "skinny" GEMM for the recurrent chain, with fused epilogues.
//
//   out[m, r] = sum_k X[m, k] * W[r, k]        m < M (batch rows), r < Rtot (weight rows)
//
// X is the concatenation along k of up to three row-major segments (the torch.cat calls at
// /root/reference/models/tts/tacotron2.py:338,:355,:360 never materialise), W is row-major
// [Rtot, Kcat] (nn.Linear / nn.LSTMCell weight layout, K-major for both operands).
//
// Mapping: one CTA = BT batch rows x R weight rows, 8 warps; the K range is split in chunks of
// KC = 16 that are dealt round-robin to the warps, each warp running its own 2-stage cp.async
// pipeline (no CTA-wide barrier in the main loop) with an (BT/8) x (R/4) register tile per lane;
// partial sums are reduced across warps through shared memory in a fixed order (deterministic),
// then the epilogue functor consumes the [R][BT] tile:
//   EpiStore     bias / addends / ReLU+Philox-dropout (Prenet, tacotron2.py:140-144)
//   EpiLstm      nn.LSTMCell pointwise (i,f,g,o; tacotron2.py:340,:357) + carried-state dropout (:341,:358)
//   EpiLstmBwd   backward of the same pointwise (BPTT, tacotron2.py:520)
#pragma once
#include "gvx_common.cuh"
#include "gvx_io.cuh"

namespace gvx {

struct Seg {
    const float *p;
    int w;    // width (multiple of 4)
    int ld;   // row stride in floats (multiple of 4)
};

struct GemmIn {
    Seg seg[3];
    int nseg;
    const float *W;
    int ldw;
    int Rtot;
    int M;
};

constexpr int GEMM_KC = 16;
constexpr int GEMM_SS = GEMM_KC + 4;   // smem row stride (floats): 80 B, conflict-free for LDS.128
constexpr int GEMM_NWARP = 8;
constexpr int GEMM_THREADS = GEMM_NWARP * 32;

template <int BT, int R>
struct GemmCfg {
    static constexpr int TB = BT / 8;
    static constexpr int RJ = R / 4;
    static constexpr int STAGE = (BT + R) * GEMM_SS;
    static constexpr int PIPE = GEMM_NWARP * 2 * STAGE;
    static constexpr int RS = BT + 8;                      // reduction row stride
    static constexpr int RED = GEMM_NWARP * R * RS;
    static constexpr int SMEM_FLOATS = PIPE > RED ? PIPE : RED;
    static constexpr size_t SMEM_BYTES = (size_t)SMEM_FLOATS * sizeof(float);
};

// ------------------------------------------------------------------ epilogues
struct EpiStore {
    float *out;
    int ldo;
    const float *bias;     // [Rtot] or null
    const float *add1;     // optional [M, Rtot] addends
    int ld1;
    const float *add2;
    int ld2;
    int mode;              // 0 plain, 1 ReLU + dropout (prenet)
    DropCfg drop;
    uint32_t site;
    int t0;                // Philox t of the first frame
    int rows_per_frame;    // rows of X per frame (B); row m -> frame m / B, batch row m % B
    int row_offset;
    // optional per batch row (continuous batching): Philox t = row_frame[brow] instead of t0 + f, row = row_id[brow] + row_offset
    const int *row_frame, *row_id;
    BfDsts bf;             // optional bf16 copies (bf16 mode), addressed by (frame, batch row, column)

    template <int BT, int R>
    __device__ __forceinline__ void run(const float *tile, int m0, int r0, int M, int Rtot) const {
        constexpr int RS = GemmCfg<BT, R>::RS;
        for (int idx = threadIdx.x; idx < R * BT; idx += GEMM_THREADS) {
            const int r = idx % R, b = idx / R;
            const int m = m0 + b, rr = r0 + r;
            if (m >= M || rr >= Rtot) continue;
            float v = tile[r * RS + b];
            if (bias) v += bias[rr];
            if (add1) v += add1[(size_t)m * ld1 + rr];
            if (add2) v += add2[(size_t)m * ld2 + rr];
            if (mode == 1) {
                const int f = m / rows_per_frame, brow = m - f * rows_per_frame;
                const uint32_t tf = row_frame ? (uint32_t)row_frame[brow] : (uint32_t)(t0 + f);
                const uint32_t rw = (uint32_t)((row_id ? row_id[brow] : brow) + row_offset);
                v = fmaxf(v, 0.f) * drop_mult(drop, site, tf, rw, (uint32_t)rr);
            }
            out[(size_t)m * ldo + rr] = v;
            if (bf.n) {
                const int f = m / rows_per_frame;
                bf_store1_t(bf, f, m - f * rows_per_frame, rr, v);
            }
        }
    }
};

// weight rows are packed unit-major: row = 4*unit + gate, gate order i,f,g,o
struct EpiLstm {
    const float *bias;      // [4*HID] packed order (b_ih + b_hh)
    const float *c_prev;    // [M, HID]
    float *c_out;           // [M, HID]
    float *h_out;           // [M, ldh] (dropped hidden, the carried state)
    int ldh;
    float *gates_out;       // [M, 4*HID] activations, or null
    DropCfg drop;
    uint32_t site;
    uint32_t t;
    int row_offset;
    int HID;

    template <int BT, int R>
    __device__ __forceinline__ void run(const float *tile, int m0, int r0, int M, int Rtot) const {
        constexpr int RS = GemmCfg<BT, R>::RS;
        constexpr int U = R / 4;
        for (int idx = threadIdx.x; idx < U * BT; idx += GEMM_THREADS) {
            const int u = idx % U, b = idx / U;
            const int m = m0 + b, row = r0 + 4 * u;
            if (m >= M || row >= Rtot) continue;
            const int unit = row >> 2;
            const float pi = tile[(4 * u + 0) * RS + b] + bias[row + 0];
            const float pf = tile[(4 * u + 1) * RS + b] + bias[row + 1];
            const float pg = tile[(4 * u + 2) * RS + b] + bias[row + 2];
            const float po = tile[(4 * u + 3) * RS + b] + bias[row + 3];
            const float gi = sigmoidf_(pi), gf = sigmoidf_(pf), gg = tanhf(pg), go = sigmoidf_(po);
            const float cn = gf * c_prev[(size_t)m * HID + unit] + gi * gg;
            float h = go * tanhf(cn);
            h *= drop_mult(drop, site, t, (uint32_t)(m + row_offset), (uint32_t)unit);
            c_out[(size_t)m * HID + unit] = cn;
            h_out[(size_t)m * ldh + unit] = h;
            if (gates_out) {
                float4 ga = make_float4(gi, gf, gg, go);
                *reinterpret_cast<float4 *>(gates_out + (size_t)m * 4 * HID + row) = ga;
            }
        }
    }
};

// d(pre-activations) of one LSTM cell from d(h_dropped) and the carried d(c)
__device__ __forceinline__ float4 lstm_bwd_point(float dh_dropped, float mult, float4 ga, float c_prev, float c_new,
                                                 float dc_in, float &dc_prev) {
    const float dh = dh_dropped * mult;
    const float tc = tanhf(c_new);
    const float d_o = dh * tc;
    const float dc = dc_in + dh * ga.w * (1.f - tc * tc);
    const float d_i = dc * ga.z, d_g = dc * ga.x, d_f = dc * c_prev;
    dc_prev = dc * ga.y;
    float4 r;
    r.x = d_i * ga.x * (1.f - ga.x);
    r.y = d_f * ga.y * (1.f - ga.y);
    r.z = d_g * (1.f - ga.z * ga.z);
    r.w = d_o * ga.w * (1.f - ga.w);
    return r;
}

// out rows are hidden units: d h_dropped[m, unit] = acc + add1 + add2, then LSTM pointwise backward
struct EpiLstmBwd {
    const float *add1;
    int ld1;
    const float *add2;
    int ld2;
    DropCfg drop;
    uint32_t site;
    uint32_t t;
    int row_offset;
    const float *gates;    // [M, 4*HID]
    const float *c_prev;   // [M, HID]
    const float *c_new;    // [M, HID]
    float *dc;             // [M, HID] carried, in/out
    float *dgates;         // [M, 4*HID]
    int HID;

    template <int BT, int R>
    __device__ __forceinline__ void run(const float *tile, int m0, int r0, int M, int Rtot) const {
        constexpr int RS = GemmCfg<BT, R>::RS;
        for (int idx = threadIdx.x; idx < R * BT; idx += GEMM_THREADS) {
            const int r = idx % R, b = idx / R;
            const int m = m0 + b, unit = r0 + r;
            if (m >= M || unit >= Rtot) continue;
            float dh = tile[r * RS + b];
            if (add1) dh += add1[(size_t)m * ld1 + unit];
            if (add2) dh += add2[(size_t)m * ld2 + unit];
            const float mult = drop_mult(drop, site, t, (uint32_t)(m + row_offset), (uint32_t)unit);
            const float4 ga = *reinterpret_cast<const float4 *>(gates + (size_t)m * 4 * HID + 4 * unit);
            float dcp;
            const float4 dp = lstm_bwd_point(dh, mult, ga, c_prev[(size_t)m * HID + unit], c_new[(size_t)m * HID + unit],
                                             dc[(size_t)m * HID + unit], dcp);
            dc[(size_t)m * HID + unit] = dcp;
            *reinterpret_cast<float4 *>(dgates + (size_t)m * 4 * HID + 4 * unit) = dp;
        }
    }
};

// ------------------------------------------------------------------ kernel
template <int BT, int R, class Epi>
__global__ void __launch_bounds__(GEMM_THREADS, 1) k_gemm(const GemmIn g, const Epi epi) {
    pdl_trigger();
    pdl_wait();
    using C = GemmCfg<BT, R>;
    constexpr int TB = C::TB, RJ = C::RJ, SS = GEMM_SS, KC = GEMM_KC;
    extern __shared__ __align__(16) float smem[];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int tb = lane & 7, tr = lane >> 3;
    const int r0 = blockIdx.x * R, m0 = blockIdx.y * BT;

    const int w0 = g.seg[0].w, w1 = g.nseg > 1 ? g.seg[1].w : 0, w2 = g.nseg > 2 ? g.seg[2].w : 0;
    const int nch0 = (w0 + KC - 1) / KC, nch1 = (w1 + KC - 1) / KC, nch2 = (w2 + KC - 1) / KC;
    const int nch = nch0 + nch1 + nch2;

    float acc[TB][RJ];
#pragma unroll
    for (int i = 0; i < TB; ++i)
#pragma unroll
        for (int j = 0; j < RJ; ++j) acc[i][j] = 0.f;

    float *mybuf = smem + wid * 2 * C::STAGE;

    auto issue = [&](int c, float *buf) {
        const float *sp;
        int sw, sld, wcol, cc = c;
        if (cc < nch0) {
            sp = g.seg[0].p; sw = w0; sld = g.seg[0].ld; wcol = 0;
        } else if (cc < nch0 + nch1) {
            cc -= nch0; sp = g.seg[1].p; sw = w1; sld = g.seg[1].ld; wcol = w0;
        } else {
            cc -= nch0 + nch1; sp = g.seg[2].p; sw = w2; sld = g.seg[2].ld; wcol = w0 + w1;
        }
        const int k0 = cc * KC;
        wcol += k0;
#pragma unroll
        for (int i = 0; i < (BT * 4) / 32; ++i) {
            const int idx = lane + 32 * i, row = idx >> 2, q = idx & 3;
            const bool ok = (m0 + row < g.M) && (k0 + q * 4 < sw);
            const float *src = ok ? sp + (size_t)(m0 + row) * sld + k0 + q * 4 : g.W;
            cp_async16(buf + row * SS + q * 4, src, ok);
        }
#pragma unroll
        for (int i = 0; i < (R * 4 + 31) / 32; ++i) {
            const int idx = lane + 32 * i, row = idx >> 2, q = idx & 3;
            if (idx < R * 4) {
                const bool ok = (r0 + row < g.Rtot) && (k0 + q * 4 < sw);
                const float *src = ok ? g.W + (size_t)(r0 + row) * g.ldw + wcol + q * 4 : g.W;
                cp_async16(buf + (BT + row) * SS + q * 4, src, ok);
            }
        }
    };

    int st = 0;
    if (wid < nch) issue(wid, mybuf);
    cp_async_commit();
    for (int c = wid; c < nch; c += GEMM_NWARP) {
        const int cn = c + GEMM_NWARP;
        if (cn < nch) issue(cn, mybuf + (st ^ 1) * C::STAGE);
        cp_async_commit();
        cp_async_wait<1>();
        __syncwarp();
        const float *As = mybuf + st * C::STAGE;
        const float *Ws = As + BT * SS;
#pragma unroll
        for (int kk = 0; kk < KC / 4; ++kk) {
            float4 a[TB];
#pragma unroll
            for (int i = 0; i < TB; ++i) a[i] = *reinterpret_cast<const float4 *>(As + (tb + 8 * i) * SS + kk * 4);
#pragma unroll
            for (int j = 0; j < RJ; ++j) {
                const float4 w = *reinterpret_cast<const float4 *>(Ws + (tr + 4 * j) * SS + kk * 4);
#pragma unroll
                for (int i = 0; i < TB; ++i) {
                    float s = acc[i][j];
                    s = fmaf(a[i].x, w.x, s);
                    s = fmaf(a[i].y, w.y, s);
                    s = fmaf(a[i].z, w.z, s);
                    s = fmaf(a[i].w, w.w, s);
                    acc[i][j] = s;
                }
            }
        }
        __syncwarp();
        st ^= 1;
    }
    cp_async_wait<0>();
    __syncthreads();

    // cross-warp reduction, fixed order (deterministic)
    float *red = smem;
#pragma unroll
    for (int i = 0; i < TB; ++i)
#pragma unroll
        for (int j = 0; j < RJ; ++j) red[(wid * R + tr + 4 * j) * C::RS + tb + 8 * i] = acc[i][j];
    __syncthreads();
    for (int idx = tid; idx < R * BT; idx += GEMM_THREADS) {
        const int r = idx / BT, b = idx % BT;
        float s = red[r * C::RS + b];
#pragma unroll
        for (int w = 1; w < GEMM_NWARP; ++w) s += red[(w * R + r) * C::RS + b];
        red[r * C::RS + b] = s;
    }
    __syncthreads();
    epi.template run<BT, R>(red, m0, r0, g.M, g.Rtot);
}

template <int BT, int R, class Epi>
inline int launch_gemm_t(const GemmIn &g, const Epi &epi, cudaStream_t stream) {
    using C = GemmCfg<BT, R>;
    static bool configured = false;
    if (!configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_gemm<BT, R, Epi>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM_BYTES));
        configured = true;
    }
    dim3 grid((g.Rtot + R - 1) / R, (g.M + BT - 1) / BT);
    GVX_CUDA(launch_pdl(k_gemm<BT, R, Epi>, grid, dim3(GEMM_THREADS), C::SMEM_BYTES, stream, g, epi));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

// R = rows of W per CTA (8 for small outputs on the critical path, 32 otherwise)
template <int R, class Epi>
inline int launch_gemm(const GemmIn &g, const Epi &epi, cudaStream_t stream) {
    GVX_CHECK(g.M > 0 && g.Rtot > 0, "empty GEMM");
    for (int s = 0; s < g.nseg; ++s) {
        GVX_CHECK(g.seg[s].w % 4 == 0 && g.seg[s].ld % 4 == 0, "GEMM segment width/stride must be a multiple of 4");
        GVX_CHECK(((uintptr_t)g.seg[s].p & 15) == 0, "GEMM segment pointer must be 16-byte aligned");
    }
    GVX_CHECK(g.ldw % 4 == 0 && ((uintptr_t)g.W & 15) == 0, "GEMM weight stride/pointer alignment");
    if (g.M <= 16) return launch_gemm_t<16, R, Epi>(g, epi, stream);
    if (g.M <= 32) return launch_gemm_t<32, R, Epi>(g, epi, stream);
    return launch_gemm_t<64, R, Epi>(g, epi, stream);
}

inline GemmIn gemm_in(const float *W, int ldw, int Rtot, int M) {
    GemmIn g;
    memset(&g, 0, sizeof(g));
    g.W = W; g.ldw = ldw; g.Rtot = Rtot; g.M = M;
    return g;
}
inline void add_seg(GemmIn &g, const float *p, int w, int ld) {
    g.seg[g.nseg].p = p; g.seg[g.nseg].w = w; g.seg[g.nseg].ld = ld;
    g.nseg++;
}

}  // namespace gvx
