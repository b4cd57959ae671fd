// genvox_b200 — bf16 mode glue around the tcgen05 gate-GEMM engine (gvx_tc.cuh).
//
// In bf16 mode (BASELINE configs[2]/[4]) the four big per-step contractions — both nn.LSTMCell gate
// GEMMs (/root/reference/models/tts/tacotron2.py:340,:357) and their BPTT transposes — plus the query
// (:98) and mel/gate projections (:361-362, inference) run on tcgen05 with bf16 operands and fp32
// accumulation.  Everything pointwise stays fp32: the engine leaves split-K fp32 partials in L2 and the
// kernels below add them (fixed order), apply the LSTM cell / its backward, and emit the next GEMM's
// operand directly in the engine's shared-memory image ([K/64][NPAD][64] bf16, SWIZZLE_128B, 16-byte vector stores)
// and, for the time-batched weight-gradient GEMMs, as row-major bf16 rows.
#pragma once
#include <cuda_bf16.h>

#include "gvx_common.cuh"
#include "gvx_gemm.cuh"
#include "gvx_io.cuh"
#include "gvx_tc.cuh"

namespace gvx {

// ------------------------------------------------------------------ LSTM cell forward from split-K partials
// partial column of (unit, gate): (unit / 32) * 128 + gate * 32 + unit % 32   (k_tc_pack_w mode 1)
struct BfLstmFwd {
    const float *P;            // [KS][B][ldp]
    int KS, ldp;
    const float *bias;         // [4*HID] unit-major (b_ih + b_hh)
    const float *c_prev;       // [B, HID]
    float *c_out;              // [B, HID]
    float *gates_out;          // [B, 4*HID] unit-major activations or null
    BfDsts h_dst;              // dropped hidden state, bf16
    DropCfg drop;
    uint32_t site, t;
    int row_offset, B, HID;
};
__global__ void __launch_bounds__(256) k_bf_lstm_fwd(const BfLstmFwd a) {
    pdl_trigger();
    pdl_wait();
    // one thread per (row, hidden unit): B*HID threads keep every SM busy; a warp covers 32 consecutive units, so
    // each partial read is one coalesced 128-byte line and the bf16 stores fill whole 16-byte image chunks
    const int total = a.B * a.HID;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int b = idx / a.HID, u = idx - b * a.HID;
        const int col = (u >> 5) * 128 + (u & 31);
        float pre[4] = {0.f, 0.f, 0.f, 0.f};
        for (int s0 = 0; s0 < a.KS; s0 += 4) {          // 16 independent loads in flight, summed in ascending split order
            float v[4][4];
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                const float *row = a.P + ((size_t)(s0 + s < a.KS ? s0 + s : s0) * a.B + b) * a.ldp + col;
#pragma unroll
                for (int g = 0; g < 4; ++g) v[s][g] = row[g * 32];
            }
#pragma unroll
            for (int s = 0; s < 4; ++s)
                if (s0 + s < a.KS) {
#pragma unroll
                    for (int g = 0; g < 4; ++g) pre[g] += v[s][g];
                }
        }
        const float4 bi = *reinterpret_cast<const float4 *>(a.bias + 4 * u);
        const float gi = sigmoidf_(pre[0] + bi.x), gf = sigmoidf_(pre[1] + bi.y);
        const float gg = tanhf(pre[2] + bi.z), go = sigmoidf_(pre[3] + bi.w);
        const float cn = gf * a.c_prev[idx] + gi * gg;
        a.c_out[idx] = cn;
        const float h = go * tanhf(cn) * drop_mult(a.drop, a.site, a.t, (uint32_t)(b + a.row_offset), (uint32_t)u);
        if (a.gates_out) *reinterpret_cast<float4 *>(a.gates_out + (size_t)b * 4 * a.HID + 4 * u) = make_float4(gi, gf, gg, go);
        bf_store1(a.h_dst, b, u, h);
    }
}

// ------------------------------------------------------------------ LSTM cell backward -> d(pre-activations) in bf16
// d h_dropped[b, u] = s0 + s1 + s2 ; outputs d gates (unit-major k = 4u + g) as engine image + row-major rows.
// Blocks past `main_blocks` compute the prenet gradient mask for frame t+1 instead:
//   dz2[b, p] = 2 * [pre2 > 0] * sum_s dpre_src[b, p]            (tacotron2.py:143)
struct BfLstmBwd {
    SrcSum s0, s1, s2;
    DropCfg drop;
    uint32_t site, t;
    int row_offset, B, HID;
    const float *gates;        // [B, 4*HID]
    const float *c_prev;       // [B, HID]
    const float *c_new;        // [B, HID]
    float *dc;                 // [B, HID] carried, in/out
    BfDsts dg_dst;             // d gates, bf16, columns 4u+g
    int main_blocks;
    SrcSum dpre_src;           // optional
    const float *pre2;         // [B, P] prenet output of that frame
    float *dz2;                // [B, P]
    int P;
};
__global__ void __launch_bounds__(256) k_bf_lstm_bwd(const BfLstmBwd a) {
    pdl_trigger();
    pdl_wait();
    if ((int)blockIdx.x >= a.main_blocks) {
        const int total = a.B * a.P;
        for (int idx = (blockIdx.x - a.main_blocks) * blockDim.x + threadIdx.x; idx < total;
             idx += (gridDim.x - a.main_blocks) * blockDim.x) {
            const int b = idx / a.P, p = idx - b * a.P;
            a.dz2[idx] = a.pre2[idx] > 0.f ? 2.f * src_get(a.dpre_src, b, p) : 0.f;
        }
        return;
    }
    // one thread per (row, hidden unit): 4 bf16 d-gates = one 8-byte store into the next GEMM's operand image
    const int total = a.B * a.HID;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += a.main_blocks * blockDim.x) {
        const int b = idx / a.HID, u = idx - b * a.HID;
        float dh = src_get(a.s0, b, u);
        if (a.s1.nsplit) dh += src_get(a.s1, b, u);
        if (a.s2.nsplit) dh += src_get(a.s2, b, u);
        const float mult = drop_mult(a.drop, a.site, a.t, (uint32_t)(b + a.row_offset), (uint32_t)u);
        const float4 ga = *reinterpret_cast<const float4 *>(a.gates + (size_t)b * 4 * a.HID + 4 * u);
        float dcp;
        const float4 dp = lstm_bwd_point(dh, mult, ga, a.c_prev[idx], a.c_new[idx], a.dc[idx], dcp);
        a.dc[idx] = dcp;
        bf_store4(a.dg_dst, b, 4 * u, make_uint2(pack_bf2(dp.x, dp.y), pack_bf2(dp.z, dp.w)));
    }
}

// out[b, m] = sum_s P[s][b][m] + bias[m]   (inference projection epilogue)
__global__ void k_bf_finalize(const float *__restrict__ P, int KS, int B, int ldp, int M, const float *__restrict__ bias,
                              float *__restrict__ out, int ldo) {
    pdl_trigger();
    pdl_wait();
    const int total = B * M;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int b = i / M, m = i - b * M;
        float s = bias ? bias[m] : 0.f;
        for (int k0 = 0; k0 < KS; k0 += 8) {           // loads first, adds after (ascending split order)
            float v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = k0 + k < KS ? P[((size_t)(k0 + k) * B + b) * ldp + m] : 0.f;
#pragma unroll
            for (int k = 0; k < 8; ++k)
                if (k0 + k < KS) s += v[k];
        }
        out[(size_t)b * ldo + m] = s;
    }
}

// fp32 -> bf16 copy of a row-major matrix (rows x cols, ld_in -> ld_out)
__global__ void k_to_bf16(const float *__restrict__ x, int ld_in, size_t rows, int cols, __nv_bfloat16 *__restrict__ y, int ld_out) {
    const size_t total = rows * cols;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / cols;
        const int c = (int)(i - r * cols);
        y[r * ld_out + c] = __float2bfloat16(x[r * ld_in + c]);
    }
}

// column sums of a row-major bf16 matrix [rows, cols]: two deterministic stages
__global__ void k_colsum_bf16_part(const __nv_bfloat16 *__restrict__ x, size_t rows, int cols, int nchunk, float *__restrict__ part) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    const int chunk = blockIdx.y;
    if (c >= cols) return;
    const size_t r0 = rows * chunk / nchunk, r1 = rows * (chunk + 1) / nchunk;
    float s = 0.f;
    for (size_t r = r0; r < r1; ++r) s += __bfloat162float(x[r * cols + c]);
    part[(size_t)chunk * cols + c] = s;
}

}  // namespace gvx
