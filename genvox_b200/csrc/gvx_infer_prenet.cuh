// genvox_b200 — both Prenet layers of one autoregressive step in ONE launch (inference, fp32 and bf16 modes).
//
// Prenet.forward (/root/reference/models/tts/tacotron2.py:140-144) on the previous mel frame is on the critical path of every
// inference step (:398): two [B x K] . [K x 256] products with ReLU and always-on dropout.  As two launches of the generic
// skinny GEMM they cost two launch + drain latencies per decoder step for 5 MFLOP.  Here 32 CTAs (8 output columns each)
// run layer 0, meet at a release/acquire grid barrier (a monotonic counter in the workspace: launch t waits for
// 32 (t + 1)), and run layer 1 on the exchanged layer-0 output.  Thread = (batch row tid & 63, column tid >> 6): the 8
// columns of a CTA are warp-uniform, so weight reads are shared-memory broadcasts and activation reads are conflict-free.
// The weights are staged before griddepcontrol.wait (they do not depend on the previous kernel of the chain); every CTA
// signals launch_dependents at once, so the next kernel of the chain can only become resident after all 32 CTAs run.
#pragma once
#include "gvx_common.cuh"
#include "gvx_io.cuh"
#include "gvx_layout.cuh"
#include "gvx_persist.cuh"

namespace gvx {

constexpr int IPN_COLS = 8;            // output columns per CTA
constexpr int IPN_THREADS = 512;       // 64 rows x 8 columns
constexpr int IPN_ROWS = 64;

struct InferPrenetArgs {
    const float *prev;                 // [B][prev_ld] previous mel frame (the go frame is all zeros)
    int prev_ld;
    const float *w0, *w1;              // [P][M], [P][P]  (state_dict layout)
    float *pre1;                       // [B][P] exchange buffer between the layers
    float *pre2;                       // [B][P] fp32 output, or null
    BfDsts bf;                         // bf16 destinations of the layer-1 output (bf16 mode)
    unsigned *bar;                     // monotonic grid-barrier counter, zero before step 0
    unsigned target;                   // gridDim.x * (t + 1)
    int *err;
    DropCfg drop;                      // p = 0.5, always on
    uint32_t t;
    int row_offset, B, M, P;
    const int *row_frame, *row_id;     // optional [B] (continuous batching): Philox t and row (before row_offset) per batch row
};

__global__ void __launch_bounds__(IPN_THREADS, 1) k_infer_prenet(const InferPrenetArgs a) {
    extern __shared__ __align__(16) float ipn_sm[];
    __shared__ int dead;
    const int M = a.M, P = a.P, B = a.B;
    const int ldx0 = M + 1, ldx1 = P + 1;
    float *w0s = ipn_sm;                                   // [8][M]
    float *w1s = w0s + ((IPN_COLS * M + 3) & ~3);          // [8][P]
    float *xs = w1s + IPN_COLS * P;                        // [64][M+1], then [64][P+1]
    float *tile = xs + IPN_ROWS * ldx1;                    // [64][8] layer-1 output tile
    const int tid = threadIdx.x, b = tid & 63, c = tid >> 6;
    const int col = blockIdx.x * IPN_COLS + c;
    pdl_trigger();
    if (tid == 0) dead = 0;
    for (int i = tid; i < IPN_COLS * M; i += IPN_THREADS) w0s[i] = a.w0[(size_t)blockIdx.x * IPN_COLS * M + i];
    for (int i = tid; i < IPN_COLS * P; i += IPN_THREADS) w1s[i] = a.w1[(size_t)blockIdx.x * IPN_COLS * P + i];
    pdl_wait();
    const int rb = b < B ? b : 0;
    const uint32_t dt = a.row_frame ? (uint32_t)a.row_frame[rb] : a.t;
    const uint32_t drow = (uint32_t)((a.row_id ? a.row_id[rb] : b) + a.row_offset);
    for (int i = tid; i < IPN_ROWS * M; i += IPN_THREADS) {
        const int r = i / M, k = i - r * M;
        xs[r * ldx0 + k] = r < B ? a.prev[(size_t)r * a.prev_ld + k] : 0.f;
    }
    __syncthreads();
    // ---- layer 0 (tacotron2.py:143, first layer)
    {
        float acc = 0.f;
        const float *xr = xs + b * ldx0, *wr = w0s + c * M;
#pragma unroll 4
        for (int k = 0; k < M; k += 4) {
            const float4 w4 = *reinterpret_cast<const float4 *>(wr + k);
            acc = fmaf(xr[k], w4.x, acc); acc = fmaf(xr[k + 1], w4.y, acc);
            acc = fmaf(xr[k + 2], w4.z, acc); acc = fmaf(xr[k + 3], w4.w, acc);
        }
        if (b < B)
            a.pre1[(size_t)b * P + col] = fmaxf(acc, 0.f) * drop_mult(a.drop, SITE_PRENET0, dt, drow, (uint32_t)col);
    }
    // ---- all 32 column slices of the layer-0 output are needed by every CTA
    __syncthreads();
    if (tid == 0) {
        gbar_arrive(a.bar);
        if (!gbar_wait(a.bar, a.target, &dead, a.err, 51)) dead = 1;
    }
    __syncthreads();
    for (int i = tid; i < IPN_ROWS * (P / 4); i += IPN_THREADS) {
        const int r = i / (P / 4), k4 = i - r * (P / 4);
        const float4 v = r < B ? __ldcg(reinterpret_cast<const float4 *>(a.pre1 + (size_t)r * P) + k4) : make_float4(0.f, 0.f, 0.f, 0.f);
        float *d = xs + r * ldx1 + 4 * k4;
        d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
    __syncthreads();
    // ---- layer 1
    {
        float acc = 0.f;
        const float *xr = xs + b * ldx1, *wr = w1s + c * P;
#pragma unroll 8
        for (int k = 0; k < P; k += 4) {
            const float4 w4 = *reinterpret_cast<const float4 *>(wr + k);
            acc = fmaf(xr[k], w4.x, acc); acc = fmaf(xr[k + 1], w4.y, acc);
            acc = fmaf(xr[k + 2], w4.z, acc); acc = fmaf(xr[k + 3], w4.w, acc);
        }
        const float v = fmaxf(acc, 0.f) * drop_mult(a.drop, SITE_PRENET1, dt, drow, (uint32_t)col);
        if (b < B && a.pre2) a.pre2[(size_t)b * P + col] = v;
        tile[b * IPN_COLS + c] = v;
    }
    if (a.bf.n) {      // the CTA's 8 columns of a row are one 16-byte chunk of the bf16 operand images
        __syncthreads();
        if (tid < IPN_ROWS && tid < B) {
            const float *tr = tile + tid * IPN_COLS;
            bf_store8(a.bf, tid, blockIdx.x * IPN_COLS,
                      make_uint4(pack_bf2(tr[0], tr[1]), pack_bf2(tr[2], tr[3]), pack_bf2(tr[4], tr[5]), pack_bf2(tr[6], tr[7])));
        }
    }
}

inline bool infer_prenet_fused_ok(const Dims &d, int B) {
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("GVX_FUSED_PRENET");
        on = (e && e[0] == '0') ? 0 : 1;
    }
    // (d.M <= d.P: the shared tile is sized [64][P + 1] and layer 0 fills it as [64][M + 1])
    return on == 1 && B <= IPN_ROWS && d.M % 4 == 0 && d.M <= d.P && d.P % IPN_COLS == 0 && d.P / IPN_COLS <= 64;
}

// prev -> PRE2 (fp32, optional) and/or bf16 images; `bar` = monotonic counter zeroed before step 0, t = step index.
// row_frame / row_id (optional, device [B]): per-row Philox t and row (before row_offset) in place of t and the batch row.
inline int run_infer_prenet(const Dims &d, const gvx_weights *w, const float *prev, int prev_ld, int B, uint64_t seed, int t,
                            int row_offset, float *pre1, float *pre2, const BfDsts *bf, unsigned *bar, int *err, cudaStream_t st,
                            const int *row_frame = nullptr, const int *row_id = nullptr) {
    InferPrenetArgs a;
    memset(&a, 0, sizeof(a));
    a.prev = prev; a.prev_ld = prev_ld; a.w0 = w->prenet_w0; a.w1 = w->prenet_w1;
    a.pre1 = pre1; a.pre2 = pre2;
    if (bf) a.bf = *bf;
    const int grid = d.P / IPN_COLS;
    a.bar = bar; a.target = (unsigned)grid * (unsigned)(t + 1); a.err = err;
    a.drop = make_drop(seed, 0.5f, 1);
    a.t = (uint32_t)t; a.row_offset = row_offset; a.B = B; a.M = d.M; a.P = d.P;
    a.row_frame = row_frame; a.row_id = row_id;
    const size_t smem = ((size_t)((IPN_COLS * d.M + 3) & ~3) + (size_t)IPN_COLS * d.P + (size_t)IPN_ROWS * (d.P + 1) + IPN_ROWS * IPN_COLS) * sizeof(float);
    static size_t configured = 0;
    if (smem > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_infer_prenet, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    GVX_CUDA(launch_pdl(k_infer_prenet, dim3(grid), dim3(IPN_THREADS), smem, st, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace gvx
