// genvox_b200 — register-tiled fast path of the location-sensitive attention step for the default
// Tacotron2 attention shape (32 location filters, kernel 31, attention_dim 128; configs/models.py:10-33).
// Same maths and I/O contract as k_attention_fwd / k_attention_bwd in gvx_attention.cuh (which remain the
// generic path for other shapes); reference: tacotron2.py:48-53, :89-129, :344-353.
//
// What changes is the instruction mix.  The generic kernels spend ~2 shared-memory loads per FMA; here
//   * the location conv is a sliding window held in registers (8 outputs x 31 taps per task, one
//     broadcast LDS per tap),
//   * the location dense layer (and its transpose in backward) uses a 4-token x 4-dim register tile per
//     lane (two LDS.128 per 16 FMAs),
//   * tanh is 1 - 2 / (1 + 2^(2x log2 e)) on the SFU (abs. error ~2e-7, far below the 1e-4 parity bound),
//   * the context and its transpose use 128-bit loads of the encoder memory rows.
#pragma once
#include "gvx_attention.cuh"

namespace gvx {

constexpr int AF_F = 32, AF_KS = 31, AF_D = 128, AF_PAD = 15;
constexpr int AF_THREADS = 512, AF_WARPS = 16;

__device__ __forceinline__ float tanh_fast(float x) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));   // 2 * log2(e)
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.f));
    return fmaf(-2.f, r, 1.f);
}

struct AttnFastSmem {
    int wcat, convT, wldT, wlc, v, q, e, w, part, scratch, total;
    int NPS, NCS, nblk;
    __host__ __device__ AttnFastSmem(int N, int E) {
        nblk = (N + 7) / 8;
        NCS = nblk * 8;
        NPS = NCS + 40;                       // window reads x[n0 .. n0+39] stay in bounds
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        wcat = take(2 * NPS);
        convT = take(AF_F * NCS);
        wldT = take(AF_F * AF_D);
        wlc = take(AF_F * 2 * AF_KS);
        v = take(AF_D);
        q = take(AF_D);
        e = take(NCS);
        w = take(NCS);
        part = take(4 * E);
        scratch = take(64);
        total = o;
    }
};

template <bool WIN>
__global__ void __launch_bounds__(AF_THREADS, 1) k_attention_fwd_fast(const AttnFwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int N = a.s.N, E = a.s.E;
    const AttnFastSmem L(N, E);
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int len = a.lengths ? (int)a.lengths[b] : N;
    float *wprev_row = a.w_prev + (size_t)b * N, *cum_row = a.cum + (size_t)b * N;

    // ---- stage the small weights while the previous kernel of the chain is still running (PDL) ...
    pdl_trigger();
    for (int i = tid; i < AF_F * 2 * AF_KS; i += AF_THREADS) sm[L.wlc + i] = a.wlc[i];
    for (int i = tid; i < AF_F * AF_D / 4; i += AF_THREADS)
        reinterpret_cast<float4 *>(sm + L.wldT)[i] = reinterpret_cast<const float4 *>(a.wldT)[i];
    if (tid < AF_D) sm[L.v + tid] = a.v[tid];
    pdl_wait();
    // ---- ... then what it produced: (w_{t-1}, cum_{t-1}) with zero halo, q
    for (int i = tid; i < 2 * L.NPS; i += AF_THREADS) {
        const int c = i / L.NPS, n = i - c * L.NPS - AF_PAD;
        float x = 0.f;
        if (n >= 0 && n < N) x = c == 0 ? wprev_row[n] : cum_row[n];
        sm[L.wcat + i] = x;
    }
    if (tid < AF_D) sm[L.q + tid] = src_get(a.q, b, tid);
    __syncthreads();
    int2 win = make_int2(0, len);
    if (WIN) win = attn_window(sm + L.wcat + AF_PAD, N, len, a.win_back, a.win_fwd, sm + L.scratch);

    // ---- location conv: task = (filter f, block of 8 tokens); sliding window in registers
    for (int task = tid; task < AF_F * L.nblk; task += AF_THREADS) {
        const int f = task / L.nblk, n0 = (task - f * L.nblk) * 8;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float x[40];
            const float4 *xr = reinterpret_cast<const float4 *>(sm + L.wcat + c * L.NPS + n0);
#pragma unroll
            for (int i = 0; i < 10; ++i) {
                const float4 t4 = xr[i];
                x[4 * i] = t4.x; x[4 * i + 1] = t4.y; x[4 * i + 2] = t4.z; x[4 * i + 3] = t4.w;
            }
            const float *wr = sm + L.wlc + (f * 2 + c) * AF_KS;
#pragma unroll
            for (int k = 0; k < AF_KS; ++k) {
                const float wk = wr[k];
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[j] = fmaf(wk, x[j + k], acc[j]);
            }
        }
        float4 *dst = reinterpret_cast<float4 *>(sm + L.convT + f * L.NCS + n0);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
    __syncthreads();
    if (a.conv_stash) {   // [N, F] rows for the backward post-pass
        float *cs = a.conv_stash + (size_t)b * N * AF_F;
        for (int i = tid; i < N * AF_F; i += AF_THREADS) {
            const int n = i >> 5, f = i & 31;
            cs[i] = sm[L.convT + f * L.NCS + n];
        }
    }

    // ---- energies: a warp takes 4 tokens at a time, each lane owns 4 attention dims
    {
        const float4 q4 = *reinterpret_cast<const float4 *>(sm + L.q + lane * 4);
        const float4 v4 = *reinterpret_cast<const float4 *>(sm + L.v + lane * 4);
        const float *pm_b = a.pm + (size_t)b * N * AF_D;
        const int ngrp = (N + 3) / 4;
        for (int grp = wid; grp < ngrp; grp += AF_WARPS) {
            const int n0 = grp * 4;
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
#pragma unroll 8
            for (int f = 0; f < AF_F; ++f) {
                const float4 wd = *reinterpret_cast<const float4 *>(sm + L.wldT + f * AF_D + lane * 4);
                const float4 c4 = *reinterpret_cast<const float4 *>(sm + L.convT + f * L.NCS + n0);
                const float cj[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    acc[j][0] = fmaf(cj[j], wd.x, acc[j][0]);
                    acc[j][1] = fmaf(cj[j], wd.y, acc[j][1]);
                    acc[j][2] = fmaf(cj[j], wd.z, acc[j][2]);
                    acc[j][3] = fmaf(cj[j], wd.w, acc[j][3]);
                }
            }
            float part[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + j;
                part[j] = 0.f;
                if (n < N) {
                    const float4 p = *reinterpret_cast<const float4 *>(pm_b + (size_t)n * AF_D + lane * 4);
                    float4 th;
                    th.x = tanh_fast((q4.x + acc[j][0]) + p.x);
                    th.y = tanh_fast((q4.y + acc[j][1]) + p.y);
                    th.z = tanh_fast((q4.z + acc[j][2]) + p.z);
                    th.w = tanh_fast((q4.w + acc[j][3]) + p.w);
                    if (a.th_stash) *reinterpret_cast<float4 *>(a.th_stash + ((size_t)b * N + n) * AF_D + lane * 4) = th;
                    part[j] = fmaf(v4.x, th.x, fmaf(v4.y, th.y, fmaf(v4.z, th.z, v4.w * th.w)));
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int j = 0; j < 4; ++j) part[j] += __shfl_xor_sync(0xffffffffu, part[j], o);
            }
            if (lane < 4) {
                const int n = n0 + lane;
                const float pv = lane == 0 ? part[0] : (lane == 1 ? part[1] : (lane == 2 ? part[2] : part[3]));
                if (n < N) sm[L.e + n] = (WIN ? n >= win.x && n < win.y : n < len) ? pv : -INFINITY;
            }
        }
    }
    __syncthreads();

    // ---- masked softmax over tokens, state update
    float mx = -INFINITY;
    for (int n = tid; n < N; n += AF_THREADS) mx = fmaxf(mx, sm[L.e + n]);
    mx = block_max(mx, sm + L.scratch);
    float sum = 0.f;
    for (int n = tid; n < N; n += AF_THREADS) {
        const float p = expf(sm[L.e + n] - mx);
        sm[L.w + n] = p;
        sum += p;
    }
    sum = block_sum(sum, sm + L.scratch);
    for (int n = tid; n < N; n += AF_THREADS) {
        const float w = sm[L.w + n] / sum;
        sm[L.w + n] = w;
        const float c_old = cum_row[n];
        a.align_out[(size_t)b * a.align_bstride + n] = w;
        if (a.cum_stash) a.cum_stash[(size_t)b * a.align_bstride + n] = c_old;
        wprev_row[n] = w;
        cum_row[n] = c_old + w;
    }
    __syncthreads();

    // ---- context: 4 token groups x 128-bit columns of memory[b], then a fixed-order reduction
    {
        const float *mem_b = a.memory + (size_t)b * N * E;
        const int tg = tid >> 7, te = tid & 127;
        for (int e4 = te * 4; e4 < E; e4 += 512) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int n = tg; n < len; n += 4) {
                const float w = sm[L.w + n];
                const float4 m = *reinterpret_cast<const float4 *>(mem_b + (size_t)n * E + e4);
                acc.x = fmaf(w, m.x, acc.x); acc.y = fmaf(w, m.y, acc.y); acc.z = fmaf(w, m.z, acc.z); acc.w = fmaf(w, m.w, acc.w);
            }
            *reinterpret_cast<float4 *>(sm + L.part + tg * E + e4) = acc;
        }
        __syncthreads();
        for (int e = tid; e < E; e += AF_THREADS) {
            const float cx = (sm[L.part + e] + sm[L.part + E + e]) + (sm[L.part + 2 * E + e] + sm[L.part + 3 * E + e]);
            if (a.ctx_out) a.ctx_out[(size_t)b * a.ctx_ld + e] = cx;
            if (a.ctx_bf.n) bf_store1(a.ctx_bf, b, e, cx);
        }
    }
}

// ------------------------------------------------------------------------------------ backward
struct AttnBwdFastSmem {
    int dctx, w, de, v, wld4, wlc, dsb, dconvT, dq, part, scratch, total;
    int NCS, NDS, nblk;
    __host__ __device__ AttnBwdFastSmem(int N, int E) {
        nblk = (N + 7) / 8;
        NCS = nblk * 8;
        NDS = NCS + 40;                        // d conv rows: index n + 15, window reads [m0, m0 + 39]
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        dctx = take(E);
        w = take(NCS);
        de = take(NCS);
        v = take(AF_D);
        wld4 = take(AF_D * AF_F);
        wlc = take(AF_F * 2 * AF_KS);
        dsb = take(AF_WARPS * 4 * AF_D);
        dconvT = take(AF_F * NDS);
        dq = take(AF_WARPS * AF_D);
        part = take(8 * 2 * NCS);
        scratch = take(64);
        total = o;
    }
};

__global__ void __launch_bounds__(AF_THREADS, 1) k_attention_bwd_fast(const AttnBwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    const int N = a.s.N, E = a.s.E;
    const AttnBwdFastSmem L(N, E);
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int len = a.lengths ? (int)a.lengths[b] : N;

    pdl_trigger();                                             // weights first (PDL prologue), then dependent data
    if (tid < AF_D) sm[L.v + tid] = a.v[tid];
    for (int i = tid; i < AF_D * AF_F; i += AF_THREADS) {      // wld [D, F] -> [D/4][F][4]
        const int d = i >> 5, f = i & 31;
        sm[L.wld4 + ((d >> 2) * AF_F + f) * 4 + (d & 3)] = a.wld[i];
    }
    for (int i = tid; i < AF_F * 2 * AF_KS; i += AF_THREADS) sm[L.wlc + i] = a.wlc[i];
    for (int i = tid; i < AF_F * L.NDS; i += AF_THREADS) sm[L.dconvT + i] = 0.f;
    pdl_wait();
    for (int e = tid; e < E; e += AF_THREADS) {
        float x = src_get(a.dctx1, b, e);
        if (a.dctx2.nsplit) x += src_get(a.dctx2, b, e);
        if (a.dctx3.nsplit) x += src_get(a.dctx3, b, e);
        sm[L.dctx + e] = x;
        a.dctx_out[(size_t)b * E + e] = x;
    }
    for (int n = tid; n < L.NCS; n += AF_THREADS) sm[L.w + n] = n < N ? a.w_t[(size_t)b * a.w_bstride + n] : 0.f;
    __syncthreads();

    // ---- d w[n] = <d ctx, memory[n]> + carried terms
    {
        const float *mem_b = a.memory + (size_t)b * N * E;
        for (int n = wid; n < L.NCS; n += AF_WARPS) {
            float dw = 0.f;
            if (n < len) {
                float part = 0.f;
                for (int e = lane * 4; e < E; e += 128) {
                    const float4 m = *reinterpret_cast<const float4 *>(mem_b + (size_t)n * E + e);
                    const float4 g = *reinterpret_cast<const float4 *>(sm + L.dctx + e);
                    part = fmaf(m.x, g.x, part); part = fmaf(m.y, g.y, part);
                    part = fmaf(m.z, g.z, part); part = fmaf(m.w, g.w, part);
                }
                part = warp_sum(part);
                dw = part + a.dw_carry[(size_t)b * N + n] + a.dcum_carry[(size_t)b * N + n];
                if (a.d_align) dw += a.d_align[(size_t)b * a.da_bstride + n];
            }
            if (lane == 0) sm[L.de + n] = dw;
        }
    }
    __syncthreads();
    // ---- softmax backward
    {
        float part = 0.f;
        for (int n = tid; n < N; n += AF_THREADS) part = fmaf(sm[L.w + n], sm[L.de + n], part);
        const float dot = block_sum(part, sm + L.scratch);
        for (int n = tid; n < L.NCS; n += AF_THREADS) {
            const float de = n < N ? sm[L.w + n] * (sm[L.de + n] - dot) : 0.f;
            sm[L.de + n] = de;
            if (n < N) a.de_out[(size_t)b * N + n] = de;
        }
    }
    __syncthreads();

    // ---- d s = d e * v * (1 - th^2);  d q += d s;  d conv[f, n] = sum_d d s[n, d] * Wld[d, f]  (4 tokens per warp pass)
    {
        const float4 v4 = *reinterpret_cast<const float4 *>(sm + L.v + lane * 4);
        float4 dqa = make_float4(0.f, 0.f, 0.f, 0.f);
        float *dsb = sm + L.dsb + wid * 4 * AF_D;
        const int ngrp = L.NCS / 4;
        for (int grp = wid; grp < ngrp; grp += AF_WARPS) {
            const int n0 = grp * 4;
            if (n0 >= len) {    // whole group masked: d conv stays zero
                if (n0 < N) {
                    for (int j = 0; j < 4; ++j)
                        if (n0 + j < N) a.dconv_out[((size_t)b * N + n0 + j) * AF_F + lane] = 0.f;
                }
                continue;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + j;
                float4 ds = make_float4(0.f, 0.f, 0.f, 0.f);
                if (n < len) {
                    const float de = sm[L.de + n];
                    const float4 th = *reinterpret_cast<const float4 *>(a.th + ((size_t)b * N + n) * AF_D + lane * 4);
                    ds.x = de * v4.x * (1.f - th.x * th.x);
                    ds.y = de * v4.y * (1.f - th.y * th.y);
                    ds.z = de * v4.z * (1.f - th.z * th.z);
                    ds.w = de * v4.w * (1.f - th.w * th.w);
                    dqa.x += ds.x; dqa.y += ds.y; dqa.z += ds.z; dqa.w += ds.w;
                }
                *reinterpret_cast<float4 *>(dsb + j * AF_D + lane * 4) = ds;
            }
            __syncwarp();
            float acc[4] = {0.f, 0.f, 0.f, 0.f};      // lane = filter f
#pragma unroll 8
            for (int dq = 0; dq < AF_D / 4; ++dq) {
                const float4 w4 = *reinterpret_cast<const float4 *>(sm + L.wld4 + (dq * AF_F + lane) * 4);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float4 x = *reinterpret_cast<const float4 *>(dsb + j * AF_D + dq * 4);
                    acc[j] = fmaf(x.x, w4.x, fmaf(x.y, w4.y, fmaf(x.z, w4.z, fmaf(x.w, w4.w, acc[j]))));
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int n = n0 + j;
                if (n < N) {
                    sm[L.dconvT + lane * L.NDS + n + AF_PAD] = acc[j];
                    a.dconv_out[((size_t)b * N + n) * AF_F + lane] = acc[j];
                }
            }
            __syncwarp();
        }
        *reinterpret_cast<float4 *>(sm + L.dq + wid * AF_D + lane * 4) = dqa;
    }
    __syncthreads();
    if (tid < AF_D) {
        float q = 0.f;
#pragma unroll
        for (int w = 0; w < AF_WARPS; ++w) q += sm[L.dq + w * AF_D + tid];
        if (a.dq_out) a.dq_out[(size_t)b * AF_D + tid] = q;
        if (a.dq_bf.n) bf_store1(a.dq_bf, b, tid, q);
    }

    // ---- d wcat[c, m] = sum_{f,k} Wlc[f,c,k] * d conv[f, m - k + pad]: task = (channel, 8 outputs, 4 filters)
    {
        const int ntask = 2 * L.nblk * 8;
        for (int task = tid; task < ntask; task += AF_THREADS) {
            const int fg = task & 7, rest = task >> 3;
            const int c = rest / L.nblk, m0 = (rest - c * L.nblk) * 8;
            float acc[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll 1
            for (int ff = 0; ff < 4; ++ff) {
                const int f = fg * 4 + ff;
                float x[40];
                const float4 *xr = reinterpret_cast<const float4 *>(sm + L.dconvT + f * L.NDS + m0);
#pragma unroll
                for (int i = 0; i < 10; ++i) {
                    const float4 t4 = xr[i];
                    x[4 * i] = t4.x; x[4 * i + 1] = t4.y; x[4 * i + 2] = t4.z; x[4 * i + 3] = t4.w;
                }
                const float *wr = sm + L.wlc + (f * 2 + c) * AF_KS;
#pragma unroll
                for (int k = 0; k < AF_KS; ++k) {
                    const float wk = wr[k];
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[j] = fmaf(wk, x[j - k + 30], acc[j]);
                }
            }
            float4 *dst = reinterpret_cast<float4 *>(sm + L.part + (fg * 2 + c) * L.NCS + m0);
            dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
            dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
    }
    __syncthreads();
    for (int idx = tid; idx < 2 * N; idx += AF_THREADS) {
        const int c = idx / N, m = idx - c * N;
        float s = 0.f;
#pragma unroll
        for (int fg = 0; fg < 8; ++fg) s += sm[L.part + (fg * 2 + c) * L.NCS + m];
        if (c == 0) a.dw_carry[(size_t)b * N + m] = s;
        else a.dcum_carry[(size_t)b * N + m] += s;
    }
}

inline bool attention_fast_ok(const AttnShape &s) {
    return s.F == AF_F && s.KS == AF_KS && s.D == AF_D && s.E % 4 == 0 && s.N >= 1;
}

template <bool WIN>
inline int launch_attention_fwd_fast_k(const AttnFwdArgs &a, size_t bytes, cudaStream_t stream) {
    static size_t configured = 0;      // per instantiation
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_fwd_fast<WIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_fwd_fast<WIN>, dim3(a.s.B), dim3(AF_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

inline int launch_attention_fwd_any(const AttnFwdArgs &a, cudaStream_t stream) {
    const AttnFastSmem L(a.s.N, a.s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    if (!attention_fast_ok(a.s) || bytes > 200 * 1024) return launch_attention_fwd(a, stream);
    return a.win_fwd ? launch_attention_fwd_fast_k<true>(a, bytes, stream) : launch_attention_fwd_fast_k<false>(a, bytes, stream);
}

inline int launch_attention_bwd_any(const AttnBwdArgs &a, cudaStream_t stream) {
    const AttnBwdFastSmem L(a.s.N, a.s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    if (!attention_fast_ok(a.s) || bytes > 200 * 1024) return launch_attention_bwd(a, stream);
    static size_t configured = 0;
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_bwd_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_bwd_fast, dim3(a.s.B), dim3(AF_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace gvx
