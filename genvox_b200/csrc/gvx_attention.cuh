// genvox_b200 — location-sensitive attention step, forward and backward.
//
// Forward = LocationLayer.forward (/root/reference/models/tts/tacotron2.py:48-53),
// Attention.get_alignment_energies (:89-104), Attention.forward (:106-129) and the cumulative
// update in Decoder.decode (:344,:353), fused in one kernel: one CTA per batch row.
//   conv[f,n]  = sum_{c,k} Wlc[f,c,k] * wcat[c, n+k-pad]          wcat = (w_{t-1}, cum_{t-1})
//   loc[n,d]   = sum_f Wld[d,f] * conv[f,n]
//   e[n]       = sum_d v[d] * tanh(q[d] + loc[n,d] + pm[n,d]);   e[n >= len] = -inf
//   w          = softmax_n(e);   ctx[e] = sum_n w[n] * memory[n,e];   cum += w
// Backward recomputes conv / loc / tanh from the stashed (w_{t-1}, cum_{t-1}, q) instead of
// saving the [N, D] activations (SURVEY.md §5: 1168*N bytes per sample-step in the reference).
#pragma once
#include <cuda_bf16.h>
#include "gvx_common.cuh"
#include "gvx_io.cuh"

namespace gvx {

constexpr int ATT_THREADS = 512;

struct AttnShape {
    int B, N, D, E, F, KS;
};

// forward shared-memory carve-up (floats)
struct AttnSmem {
    int wcat, conv, wldT, wlc, v, q, e, w, scratch, total;
    __host__ __device__ AttnSmem(const AttnShape &s) {
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        wcat = take(2 * (s.N + s.KS - 1));
        conv = take(s.N * (s.F + 1));
        wldT = take(s.F * s.D);
        wlc = take(s.F * 2 * s.KS);
        v = take(s.D);
        q = take(s.D);
        e = take(s.N);
        w = take(s.N);
        scratch = take(64);
        total = o;
    }
};

struct AttnFwdArgs {
    AttnShape s;
    SrcSum q;                // [B, D] processed query (possibly split-K partials)
    const float *pm;         // [B, N, D]
    const float *memory;     // [B, N, E]
    const float *wlc;        // [F, 2, KS]
    const float *wldT;       // [F, D]  (location_dense weight, transposed copy from the packed weights)
    const float *v;          // [D]
    const int64_t *lengths;  // [B] or null
    float *w_prev;           // [B, N] in/out
    float *cum;              // [B, N] in/out
    float *align_out;        // row b at align_out + b * align_bstride
    long long align_bstride;
    float *cum_stash;        // cum before the update, same addressing as align_out; or null
    float *ctx_out;          // [B, ctx_ld] fp32, or null
    int ctx_ld;
    BfDsts ctx_bf;           // bf16 copies of the context (bf16 mode)
    float *th_stash;         // [B, N, D] tanh(q + loc + pm) for the backward pass, or null
    float *conv_stash;       // [B, N, F] location-conv output for the backward pass, or null
    int th_bf16;             // k_attention_fwd_c2 only: write th_stash as bf16 rows of 256 B with 16-byte chunks swizzled by (token & 7),
                             // the format the persistent BPTT chain reads (gvx_fused_bwd.cuh)
    int win_back, win_fwd;   // attention constraint (inference): win_fwd == 0 off, else attend only to
                             // [last - win_back, last + win_fwd), last = argmax of w_prev's row (attn_window).  The forward
                             // kernels are instantiated for WIN = (win_fwd != 0), so the unconstrained code is unchanged
};

// The token window [lo, hi) a constrained step may attend to: last = argmax_n w[n] (lowest index on ties, as torch.argmax),
// lo = max(0, last - back), hi = min(len, last + fwd).  It is never empty: last lies in the previous step's window.
// A block reduction of (value, ~index) keys; every thread gets the result.  `scratch`: 64 floats, 8-byte aligned.
__device__ __forceinline__ int2 attn_window(const float *w, int N, int len, int back, int fwd, float *scratch) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    unsigned long long best = 0;
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        const unsigned u = __float_as_uint(w[n]);
        const unsigned key = (u & 0x80000000u) ? ~u : (u | 0x80000000u);       // order-preserving map of the float
        const unsigned long long k = ((unsigned long long)key << 32) | (unsigned)(~n);
        best = k > best ? k : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long k = __shfl_xor_sync(0xffffffffu, best, o);
        best = k > best ? k : best;
    }
    unsigned long long *sc = reinterpret_cast<unsigned long long *>(scratch);
    __syncthreads();
    if (lane == 0) sc[wid] = best;
    __syncthreads();
    if (wid == 0) {
        unsigned long long x = lane < nw ? sc[lane] : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long k = __shfl_xor_sync(0xffffffffu, x, o);
            x = k > x ? k : x;
        }
        if (lane == 0) sc[0] = x;          // lanes 1..31 read only sc[1..31] above
    }
    __syncthreads();
    const int last = (int)~(unsigned)(sc[0] & 0xffffffffull);
    return make_int2(max(0, last - back), fwd > len - last ? len : last + fwd);
}

// stage w_{t-1} / cum_{t-1} (zero halo), the small weights and q into shared memory
__device__ __forceinline__ void attn_stage_inputs(const AttnShape &s, const AttnSmem &L, float *sm, const float *wprev_row,
                                                  const float *cum_row, const float *wlc, const float *wldT, const float *v,
                                                  const SrcSum &q, int b) {
    const int pad = (s.KS - 1) / 2, NP = s.N + s.KS - 1;
    for (int i = threadIdx.x; i < 2 * NP; i += blockDim.x) {
        const int c = i / NP, j = i - c * NP, n = j - pad;
        float x = 0.f;
        if (n >= 0 && n < s.N) x = c == 0 ? wprev_row[n] : cum_row[n];
        sm[L.wcat + i] = x;
    }
    for (int i = threadIdx.x; i < s.F * 2 * s.KS; i += blockDim.x) sm[L.wlc + i] = wlc[i];
    for (int i = threadIdx.x; i < s.F * s.D; i += blockDim.x) sm[L.wldT + i] = wldT[i];
    for (int i = threadIdx.x; i < s.D; i += blockDim.x) {
        sm[L.v + i] = v[i];
        sm[L.q + i] = src_get(q, b, i);
    }
}

// conv[n][f] (row stride F+1) from wcat
__device__ __forceinline__ void attn_conv(const AttnShape &s, const AttnSmem &L, float *sm) {
    const int NP = s.N + s.KS - 1;
    for (int idx = threadIdx.x; idx < s.N * s.F; idx += blockDim.x) {
        const int f = idx / s.N, n = idx - f * s.N;
        const float *w0 = sm + L.wlc + (f * 2 + 0) * s.KS, *w1 = w0 + s.KS;
        const float *x0 = sm + L.wcat + n, *x1 = x0 + NP;
        float a = 0.f;
        for (int k = 0; k < s.KS; ++k) a = fmaf(w0[k], x0[k], a);
        for (int k = 0; k < s.KS; ++k) a = fmaf(w1[k], x1[k], a);
        sm[L.conv + n * (s.F + 1) + f] = a;
    }
}

template <bool WIN>
__global__ void __launch_bounds__(ATT_THREADS, 1) k_attention_fwd(const AttnFwdArgs a) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float sm[];
    const AttnShape s = a.s;
    const AttnSmem L(s);
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarp = blockDim.x >> 5;
    const int len = a.lengths ? (int)a.lengths[b] : s.N;
    float *wprev_row = a.w_prev + (size_t)b * s.N, *cum_row = a.cum + (size_t)b * s.N;

    attn_stage_inputs(s, L, sm, wprev_row, cum_row, a.wlc, a.wldT, a.v, a.q, b);
    __syncthreads();
    int2 win = make_int2(0, len);
    if (WIN) win = attn_window(sm + L.wcat + (s.KS - 1) / 2, s.N, len, a.win_back, a.win_fwd, sm + L.scratch);
    attn_conv(s, L, sm);
    __syncthreads();
    if (a.conv_stash) {
        float *cs = a.conv_stash + (size_t)b * s.N * s.F;
        for (int i = tid; i < s.N * s.F; i += blockDim.x) {
            const int n = i / s.F, f = i - n * s.F;
            cs[i] = sm[L.conv + n * (s.F + 1) + f];
        }
    }

    // energies: one warp per token, lanes own 4 consecutive d
    const float *pm_b = a.pm + (size_t)b * s.N * s.D;
    for (int n = wid; n < s.N; n += nwarp) {
        float part = 0.f;
        for (int d0 = lane * 4; d0 < s.D; d0 += 128) {
            float4 loc = make_float4(0.f, 0.f, 0.f, 0.f);
            const float *cv = sm + L.conv + n * (s.F + 1);
            for (int f = 0; f < s.F; ++f) {
                const float c = cv[f];
                const float4 wd = *reinterpret_cast<const float4 *>(sm + L.wldT + f * s.D + d0);
                loc.x = fmaf(c, wd.x, loc.x); loc.y = fmaf(c, wd.y, loc.y);
                loc.z = fmaf(c, wd.z, loc.z); loc.w = fmaf(c, wd.w, loc.w);
            }
            const float4 p = *reinterpret_cast<const float4 *>(pm_b + (size_t)n * s.D + d0);
            const float4 qq = *reinterpret_cast<const float4 *>(sm + L.q + d0);
            const float4 vv = *reinterpret_cast<const float4 *>(sm + L.v + d0);
            float4 th;
            th.x = tanhf((qq.x + loc.x) + p.x);
            th.y = tanhf((qq.y + loc.y) + p.y);
            th.z = tanhf((qq.z + loc.z) + p.z);
            th.w = tanhf((qq.w + loc.w) + p.w);
            if (a.th_stash) *reinterpret_cast<float4 *>(a.th_stash + ((size_t)b * s.N + n) * s.D + d0) = th;
            part = fmaf(vv.x, th.x, part);
            part = fmaf(vv.y, th.y, part);
            part = fmaf(vv.z, th.z, part);
            part = fmaf(vv.w, th.w, part);
        }
        part = warp_sum(part);
        if (lane == 0) sm[L.e + n] = (WIN ? n >= win.x && n < win.y : n < len) ? part : -INFINITY;
    }
    __syncthreads();

    // masked softmax over tokens
    float mx = -INFINITY;
    for (int n = tid; n < s.N; n += blockDim.x) mx = fmaxf(mx, sm[L.e + n]);
    mx = block_max(mx, sm + L.scratch);
    float sum = 0.f;
    for (int n = tid; n < s.N; n += blockDim.x) {
        const float p = expf(sm[L.e + n] - mx);
        sm[L.w + n] = p;
        sum += p;
    }
    sum = block_sum(sum, sm + L.scratch);
    for (int n = tid; n < s.N; n += blockDim.x) {
        const float w = sm[L.w + n] / sum;
        sm[L.w + n] = w;
        const float c_old = cum_row[n];
        a.align_out[(size_t)b * a.align_bstride + n] = w;
        if (a.cum_stash) a.cum_stash[(size_t)b * a.align_bstride + n] = c_old;
        wprev_row[n] = w;
        cum_row[n] = c_old + w;
    }
    __syncthreads();

    // context: ctx[e] = sum_n w[n] * memory[b, n, e]   (coalesced rows of E floats)
    const float *mem_b = a.memory + (size_t)b * s.N * s.E;
    for (int e = tid; e < s.E; e += blockDim.x) {
        float c0 = 0.f, c1 = 0.f, c2 = 0.f, c3 = 0.f;
        int n = 0;
        for (; n + 3 < len; n += 4) {
            c0 = fmaf(sm[L.w + n + 0], mem_b[(size_t)(n + 0) * s.E + e], c0);
            c1 = fmaf(sm[L.w + n + 1], mem_b[(size_t)(n + 1) * s.E + e], c1);
            c2 = fmaf(sm[L.w + n + 2], mem_b[(size_t)(n + 2) * s.E + e], c2);
            c3 = fmaf(sm[L.w + n + 3], mem_b[(size_t)(n + 3) * s.E + e], c3);
        }
        for (; n < len; ++n) c0 = fmaf(sm[L.w + n], mem_b[(size_t)n * s.E + e], c0);
        const float cx = (c0 + c1) + (c2 + c3);
        if (a.ctx_out) a.ctx_out[(size_t)b * a.ctx_ld + e] = cx;
        if (a.ctx_bf.n) bf_store1(a.ctx_bf, b, e, cx);
    }
}

template <bool WIN>
inline int launch_attention_fwd_k(const AttnFwdArgs &a, size_t bytes, cudaStream_t stream) {
    static size_t configured = 0;      // per instantiation
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_fwd<WIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_fwd<WIN>, dim3(a.s.B), dim3(ATT_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

inline int launch_attention_fwd(const AttnFwdArgs &a, cudaStream_t stream) {
    const AttnSmem L(a.s);
    const size_t bytes = (size_t)L.total * sizeof(float);
    GVX_CHECK(bytes <= 200 * 1024, "attention: token count too large for the shared-memory tile");
    GVX_CHECK(a.s.D % 4 == 0, "attention_dim must be a multiple of 4");
    return a.win_fwd ? launch_attention_fwd_k<true>(a, bytes, stream) : launch_attention_fwd_k<false>(a, bytes, stream);
}

// ------------------------------------------------------------------ backward (one step, one CTA per row)
// Sequential part of the attention BPTT only; everything that can be batched over time
// (d processed_memory, d v, d location_dense, d location_conv, d memory, d query weight) is
// computed afterwards from the stashes by the post-pass kernels in gvx_bwd.cu.
struct AttnBwdSmem {
    int dctx, w, de, v, wld4, wlc, dsbuf, dconv, dq, scratch, total;
    __host__ __device__ AttnBwdSmem(const AttnShape &s, int nwarp) {
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        dctx = take(s.E);
        w = take(s.N);
        de = take(s.N);
        v = take(s.D);
        wld4 = take(s.D * s.F);
        wlc = take(s.F * 2 * s.KS);
        dsbuf = take(nwarp * s.D);
        dconv = take((s.N + s.KS - 1) * (s.F + 1));
        dq = take(s.D);
        scratch = take(64);
        total = o;
    }
};

struct AttnBwdArgs {
    AttnShape s;
    const float *memory;       // [B, N, E]
    const float *wlc;          // [F, 2, KS]
    const float *wld;          // [D, F]
    const float *v;            // [D]
    const int64_t *lengths;
    const float *w_t;          // alignments of this step; row b at w_t + b * w_bstride
    long long w_bstride;
    const float *th;           // [B, N, D] stashed tanh
    SrcSum dctx1, dctx2, dctx3;    // d ctx_t contributions (2 and 3 may be empty)
    const float *d_align;      // upstream d alignments of this step (row stride da_bstride) or null
    long long da_bstride;
    float *dw_carry;           // [B, N] in: d w_t from step t+1's conv channel 0; out: d w_{t-1}
    float *dcum_carry;         // [B, N] in: d cum_t; out: d cum_{t-1}
    float *dctx_out;           // [B, E] total d ctx_t
    float *de_out;             // [B, N] d energies
    float *dq_out;             // [B, D] d processed query (fp32) or null
    BfDsts dq_bf;              // bf16 copies of d q (bf16 mode)
    float *dconv_out;          // [B, N, F] d conv output
    // optional (2-CTA cluster kernel only): d h_att from the query projection, dhq_out[b, u] = sum_d bf16(d q[b, d]) * WqB[d, u]
    const __nv_bfloat16 *WqB;  // [D, A] row-major bf16 W_query, or null
    float *dhq_out;            // [B, A]
    int A;
    int dctx12_static;         // 1: dctx1 / dctx2 were complete before the launch chain began (time-batched GEMMs): the cluster
                               // kernel may read them in its PDL prologue, before griddepcontrol.wait
    const __nv_bfloat16 *memb; // optional bf16 copy of `memory` [B, N, E] (2-CTA cluster kernel: operand of d w in bf16 mode)
    long long *dbg;            // optional clock64 stamps of CTA 0 (gvx_debug_timeline), row dbg_t
    int dbg_t;
};

__global__ void __launch_bounds__(ATT_THREADS, 1) k_attention_bwd(const AttnBwdArgs a) {
    pdl_trigger();
    pdl_wait();
    extern __shared__ __align__(16) float sm[];
    const AttnShape s = a.s;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nwarp = blockDim.x >> 5;
    const AttnBwdSmem L(s, nwarp);
    const int len = a.lengths ? (int)a.lengths[b] : s.N;
    const int pad = (s.KS - 1) / 2, NP = s.N + s.KS - 1;

    for (int e = tid; e < s.E; e += blockDim.x) {
        float x = src_get(a.dctx1, b, e);
        if (a.dctx2.nsplit) x += src_get(a.dctx2, b, e);
        if (a.dctx3.nsplit) x += src_get(a.dctx3, b, e);
        sm[L.dctx + e] = x;
        a.dctx_out[(size_t)b * s.E + e] = x;
    }
    for (int n = tid; n < s.N; n += blockDim.x) sm[L.w + n] = a.w_t[(size_t)b * a.w_bstride + n];
    for (int i = tid; i < s.D; i += blockDim.x) { sm[L.v + i] = a.v[i]; sm[L.dq + i] = 0.f; }
    for (int i = tid; i < s.D * s.F; i += blockDim.x) {
        const int d = i / s.F, f = i - d * s.F;
        sm[L.wld4 + ((d >> 2) * s.F + f) * 4 + (d & 3)] = a.wld[i];
    }
    for (int i = tid; i < s.F * 2 * s.KS; i += blockDim.x) sm[L.wlc + i] = a.wlc[i];
    for (int i = tid; i < NP * (s.F + 1); i += blockDim.x) sm[L.dconv + i] = 0.f;
    __syncthreads();

    // d w[n] = <d ctx, memory[n]> + carried terms
    const float *mem_b = a.memory + (size_t)b * s.N * s.E;
    for (int n = wid; n < s.N; n += nwarp) {
        float dw = 0.f;
        if (n < len) {
            float part = 0.f;
            for (int e = lane * 4; e < s.E; e += 128) {
                const float4 m = *reinterpret_cast<const float4 *>(mem_b + (size_t)n * s.E + e);
                const float4 g = *reinterpret_cast<const float4 *>(sm + L.dctx + e);
                part = fmaf(m.x, g.x, part); part = fmaf(m.y, g.y, part);
                part = fmaf(m.z, g.z, part); part = fmaf(m.w, g.w, part);
            }
            part = warp_sum(part);
            dw = part + a.dw_carry[(size_t)b * s.N + n] + a.dcum_carry[(size_t)b * s.N + n];
            if (a.d_align) dw += a.d_align[(size_t)b * a.da_bstride + n];
        }
        if (lane == 0) sm[L.de + n] = dw;
    }
    __syncthreads();
    // softmax backward: d e = w * (d w - <w, d w>)
    float part = 0.f;
    for (int n = tid; n < s.N; n += blockDim.x) part = fmaf(sm[L.w + n], sm[L.de + n], part);
    const float dot = block_sum(part, sm + L.scratch);
    for (int n = tid; n < s.N; n += blockDim.x) {
        const float de = sm[L.w + n] * (sm[L.de + n] - dot);
        sm[L.de + n] = de;
        a.de_out[(size_t)b * s.N + n] = de;
    }
    __syncthreads();

    // d s = d e * v * (1 - th^2);  d q += d s;  d conv[n, f] = sum_d d s[d] * Wld[d, f]
    float *dsb = sm + L.dsbuf + wid * s.D;
    float4 dqa[4];                       // per-warp partial of d q (D <= 512), reduced in a fixed order below
#pragma unroll
    for (int i = 0; i < 4; ++i) dqa[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int n = wid; n < s.N; n += nwarp) {
        float *dco = a.dconv_out + ((size_t)b * s.N + n) * s.F;
        if (n < len) {
            const float de = sm[L.de + n];
#pragma unroll
            for (int it = 0; it < 4; ++it) {
                const int d0 = lane * 4 + it * 128;
                if (d0 >= s.D) break;
                const float4 th = *reinterpret_cast<const float4 *>(a.th + ((size_t)b * s.N + n) * s.D + d0);
                const float4 vv = *reinterpret_cast<const float4 *>(sm + L.v + d0);
                float4 ds;
                ds.x = de * vv.x * (1.f - th.x * th.x);
                ds.y = de * vv.y * (1.f - th.y * th.y);
                ds.z = de * vv.z * (1.f - th.z * th.z);
                ds.w = de * vv.w * (1.f - th.w * th.w);
                *reinterpret_cast<float4 *>(dsb + d0) = ds;
                dqa[it].x += ds.x; dqa[it].y += ds.y; dqa[it].z += ds.z; dqa[it].w += ds.w;
            }
            __syncwarp();
            for (int f = lane; f < s.F; f += 32) {
                float acc = 0.f;
                for (int dq = 0; dq < s.D / 4; ++dq) {
                    const float4 x = *reinterpret_cast<const float4 *>(dsb + dq * 4);
                    const float4 w4 = *reinterpret_cast<const float4 *>(sm + L.wld4 + (dq * s.F + f) * 4);
                    acc = fmaf(x.x, w4.x, acc); acc = fmaf(x.y, w4.y, acc);
                    acc = fmaf(x.z, w4.z, acc); acc = fmaf(x.w, w4.w, acc);
                }
                sm[L.dconv + (n + pad) * (s.F + 1) + f] = acc;
                dco[f] = acc;
            }
            __syncwarp();
        } else {
            for (int f = lane; f < s.F; f += 32) dco[f] = 0.f;
        }
    }
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        const int d0 = lane * 4 + it * 128;
        if (d0 < s.D) *reinterpret_cast<float4 *>(dsb + d0) = dqa[it];
    }
    __syncthreads();
    for (int i = tid; i < s.D; i += blockDim.x) {
        float q = 0.f;
        for (int w = 0; w < nwarp; ++w) q += sm[L.dsbuf + w * s.D + i];
        if (a.dq_out) a.dq_out[(size_t)b * s.D + i] = q;
        if (a.dq_bf.n) bf_store1(a.dq_bf, b, i, q);
    }

    // d wcat[c, m] = sum_{f,k} Wlc[f,c,k] * d conv[m - k + pad, f]
    for (int idx = tid; idx < 2 * s.N; idx += blockDim.x) {
        const int c = idx / s.N, m = idx - c * s.N;
        float acc = 0.f;
        for (int f = 0; f < s.F; ++f) {
            const float *wk = sm + L.wlc + (f * 2 + c) * s.KS;
            const float *dc = sm + L.dconv + (m + 2 * pad) * (s.F + 1) + f;
            for (int k = 0; k < s.KS; ++k) acc = fmaf(wk[k], dc[-k * (s.F + 1)], acc);
        }
        if (c == 0) a.dw_carry[(size_t)b * s.N + m] = acc;
        else a.dcum_carry[(size_t)b * s.N + m] += acc;
    }
}

inline int launch_attention_bwd(const AttnBwdArgs &a, cudaStream_t stream) {
    const AttnBwdSmem L(a.s, ATT_THREADS / 32);
    const size_t bytes = (size_t)L.total * sizeof(float);
    GVX_CHECK(bytes <= 200 * 1024, "attention backward: token count too large for the shared-memory tile");
    GVX_CHECK(a.s.D <= 512 && a.s.D % 4 == 0 && a.s.E % 4 == 0, "attention backward: att_dim must be <= 512");
    static size_t configured = 0;
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_bwd, dim3(a.s.B), dim3(ATT_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace gvx
