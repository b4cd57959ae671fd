// genvox_b200 — attention step split over a 2-CTA thread-block cluster per batch row.
//
// With B = 64 rows one CTA per row leaves 84 of the 148 SMs idle and the kernel is latency-bound (ncu:
// issue slots 30 % busy, long-scoreboard and barrier stalls dominate).  Here the two CTAs of a cluster
// split the tokens of a row in halves and exchange, through distributed shared memory, only
//   forward : the softmax max and sum (2 floats) and the partial context (E floats),
//   backward: <w, dw> (1 float), the partial d q (D floats) and a 15-token halo of d conv.
// Maths and I/O contract are those of k_attention_fwd_fast / k_attention_bwd_fast (gvx_attention_fast.cuh);
// reference: tacotron2.py:48-53, :89-129, :344-353.  Reductions across the pair are always rank 0 + rank 1, so
// both CTAs hold bit-identical values and results do not depend on scheduling.
#pragma once
#include <cooperative_groups.h>

#include "gvx_attention_fast.cuh"

namespace gvx {

namespace cg = cooperative_groups;

struct AttnC2Geom {
    int NH;        // tokens per CTA (multiple of 8)
    int nblk;      // NH / 8
    int NPS;       // local wcat row length
    int NDS;       // local d conv row length (backward)
    __host__ __device__ explicit AttnC2Geom(int N) {
        NH = (((N + 1) / 2) + 7) & ~7;
        nblk = NH / 8;
        NPS = NH + 40;
        NDS = NH + 40;
    }
};

struct AttnC2FwdSmem {
    int wcat, convT, wldT, wlc, v, q, e, w, part, ctxp, xch, scratch, pms, total;
    __host__ __device__ AttnC2FwdSmem(int N, int E) {
        const AttnC2Geom g(N);
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        wcat = take(2 * g.NPS);
        convT = take(AF_F * g.NH);
        wldT = take(AF_F * AF_D);
        wlc = take(AF_F * 2 * AF_KS);
        v = take(AF_D);
        q = take(AF_D);
        e = take(g.NH);
        w = take(g.NH);
        part = take(4 * E);
        ctxp = take(E);        // this CTA's partial context, read by the peer
        xch = take(8);         // [0] local max, [1] local sum
        scratch = take(64);
        pms = take(g.NH * AF_D);   // processed memory of the own tokens, prefetched with cp.async in the PDL prologue
        total = o;
    }
};

template <bool WIN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(AF_THREADS, 1) k_attention_fwd_c2(const AttnFwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int N = a.s.N, E = a.s.E;
    const AttnC2Geom G(N);
    const AttnC2FwdSmem L(N, E);
    const int rank = (int)cluster.block_rank(), peer = rank ^ 1;
    const int b = blockIdx.x >> 1, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int len = a.lengths ? (int)a.lengths[b] : N;
    const int n_lo = rank * G.NH;
    const int n_own = max(0, min(N, n_lo + G.NH) - n_lo);      // valid own tokens: local index [0, n_own)
    float *wprev_row = a.w_prev + (size_t)b * N, *cum_row = a.cum + (size_t)b * N;

    pdl_trigger();
    {   // processed memory rows of the own tokens do not depend on the previous kernel: asynchronous prefetch
        const float *src = a.pm + ((size_t)b * N + n_lo) * AF_D;
        for (int i = tid; i < n_own * (AF_D / 4); i += AF_THREADS) cp_async16(sm + L.pms + i * 4, src + (size_t)i * 4, true);
        cp_async_commit();
    }
    for (int i = tid; i < AF_F * 2 * AF_KS; i += AF_THREADS) sm[L.wlc + i] = a.wlc[i];
    for (int i = tid; i < AF_F * AF_D / 4; i += AF_THREADS)
        reinterpret_cast<float4 *>(sm + L.wldT)[i] = reinterpret_cast<const float4 *>(a.wldT)[i];
    if (tid < AF_D) sm[L.v + tid] = a.v[tid];
    pdl_wait();
    // local window of (w_{t-1}, cum_{t-1}): index i <-> token n_lo + i - 15, zero outside [0, N)
    for (int i = tid; i < 2 * G.NPS; i += AF_THREADS) {
        const int c = i / G.NPS, n = n_lo + (i - c * G.NPS) - AF_PAD;
        float x = 0.f;
        if (n >= 0 && n < N) x = c == 0 ? wprev_row[n] : cum_row[n];
        sm[L.wcat + i] = x;
    }
    if (tid < AF_D) sm[L.q + tid] = src_get(a.q, b, tid);
    __syncthreads();
    // the constraint needs the argmax of the whole w_{t-1} row: both CTAs reduce it from global memory, before the first
    // cluster.sync (after it the peer overwrites its half of the row with w_t)
    int2 win = make_int2(0, len);
    if (WIN) win = attn_window(wprev_row, N, len, a.win_back, a.win_fwd, sm + L.scratch);

    // ---- location conv for the own tokens
    for (int task = tid; task < AF_F * G.nblk; task += AF_THREADS) {
        const int f = task / G.nblk, n0 = (task - f * G.nblk) * 8;
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            float x[40];
            const float4 *xr = reinterpret_cast<const float4 *>(sm + L.wcat + c * G.NPS + n0);
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
        float4 *dst = reinterpret_cast<float4 *>(sm + L.convT + f * G.NH + n0);
        dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
        dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
    }
    cp_async_wait<0>();       // the prefetched processed-memory rows have landed (each thread waits for its own copies)
    __syncthreads();
    if (a.conv_stash) {
        float *cs = a.conv_stash + ((size_t)b * N + n_lo) * AF_F;
        for (int i = tid; i < n_own * AF_F; i += AF_THREADS) {
            const int n = i >> 5, f = i & 31;
            cs[i] = sm[L.convT + f * G.NH + n];
        }
    }

    // ---- energies of the own tokens (4 tokens per warp pass, 4 attention dims per lane)
    {
        const float4 q4 = *reinterpret_cast<const float4 *>(sm + L.q + lane * 4);
        const float4 v4 = *reinterpret_cast<const float4 *>(sm + L.v + lane * 4);
        const float *pm_b = sm + L.pms;
        const int ngrp = (n_own + 3) / 4;
        for (int grp = wid; grp < ngrp; grp += AF_WARPS) {
            const int n0 = grp * 4;
            float4 p[4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
                p[j] = n0 + j < n_own ? *reinterpret_cast<const float4 *>(pm_b + (size_t)(n0 + j) * AF_D + lane * 4)
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
#pragma unroll 8
            for (int f = 0; f < AF_F; ++f) {
                const float4 wd = *reinterpret_cast<const float4 *>(sm + L.wldT + f * AF_D + lane * 4);
                const float4 c4 = *reinterpret_cast<const float4 *>(sm + L.convT + f * G.NH + n0);
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
                part[j] = 0.f;
                if (n0 + j < n_own) {
                    float4 th;
                    th.x = tanh_fast((q4.x + acc[j][0]) + p[j].x);
                    th.y = tanh_fast((q4.y + acc[j][1]) + p[j].y);
                    th.z = tanh_fast((q4.z + acc[j][2]) + p[j].z);
                    th.w = tanh_fast((q4.w + acc[j][3]) + p[j].w);
                    if (a.th_stash) {
                        const int ng = n_lo + n0 + j;
                        if (a.th_bf16)
                            *reinterpret_cast<uint2 *>(reinterpret_cast<uint8_t *>(a.th_stash) + ((size_t)b * N + ng) * (AF_D * 2) +
                                                       (((lane >> 1) ^ (ng & 7)) << 4) + (lane & 1) * 8) =
                                make_uint2(pack_bf2(th.x, th.y), pack_bf2(th.z, th.w));
                        else
                            *reinterpret_cast<float4 *>(a.th_stash + ((size_t)b * N + ng) * AF_D + lane * 4) = th;
                    }
                    part[j] = fmaf(v4.x, th.x, fmaf(v4.y, th.y, fmaf(v4.z, th.z, v4.w * th.w)));
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int j = 0; j < 4; ++j) part[j] += __shfl_xor_sync(0xffffffffu, part[j], o);
            }
            if (lane < 4) {
                const int nl = n0 + lane;
                const float pv = lane == 0 ? part[0] : (lane == 1 ? part[1] : (lane == 2 ? part[2] : part[3]));
                if (nl < n_own) sm[L.e + nl] = (WIN ? n_lo + nl >= win.x && n_lo + nl < win.y : (n_lo + nl) < len) ? pv : -INFINITY;
            }
        }
    }
    __syncthreads();

    // ---- masked softmax over ALL tokens of the row: exchange max, then sum, with the peer CTA
    float mx = -INFINITY;
    for (int n = tid; n < n_own; n += AF_THREADS) mx = fmaxf(mx, sm[L.e + n]);
    mx = block_max(mx, sm + L.scratch);
    if (tid == 0) sm[L.xch + 0] = mx;
    cluster.sync();
    const float *peer_sm = cluster.map_shared_rank(sm, peer);
    mx = fmaxf(mx, peer_sm[L.xch + 0]);
    float sum = 0.f;
    for (int n = tid; n < n_own; n += AF_THREADS) {
        const float pexp = expf(sm[L.e + n] - mx);
        sm[L.w + n] = pexp;
        sum += pexp;
    }
    sum = block_sum(sum, sm + L.scratch);
    if (tid == 0) sm[L.xch + 1] = sum;
    cluster.sync();
    {
        const float other = peer_sm[L.xch + 1];
        sum = rank == 0 ? sum + other : other + sum;       // always rank 0 + rank 1
    }
    for (int n = tid; n < n_own; n += AF_THREADS) {
        const float w = sm[L.w + n] / sum;
        sm[L.w + n] = w;
        const int ng = n_lo + n;
        const float c_old = cum_row[ng];
        a.align_out[(size_t)b * a.align_bstride + ng] = w;
        if (a.cum_stash) a.cum_stash[(size_t)b * a.align_bstride + ng] = c_old;
        wprev_row[ng] = w;
        cum_row[ng] = c_old + w;
    }
    __syncthreads();

    // ---- partial context over the own tokens, then each CTA finalises half of the E columns
    {
        const float *mem_b = a.memory + ((size_t)b * N + n_lo) * E;
        const int own_len = max(0, min(len, n_lo + n_own) - n_lo);
        const int tg = tid >> 7, te = tid & 127;
        for (int e4 = te * 4; e4 < E; e4 += 512) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int n = tg; n < own_len; n += 4) {
                const float w = sm[L.w + n];
                const float4 m = *reinterpret_cast<const float4 *>(mem_b + (size_t)n * E + e4);
                acc.x = fmaf(w, m.x, acc.x); acc.y = fmaf(w, m.y, acc.y); acc.z = fmaf(w, m.z, acc.z); acc.w = fmaf(w, m.w, acc.w);
            }
            *reinterpret_cast<float4 *>(sm + L.part + tg * E + e4) = acc;
        }
        __syncthreads();
        for (int e = tid; e < E; e += AF_THREADS)
            sm[L.ctxp + e] = (sm[L.part + e] + sm[L.part + E + e]) + (sm[L.part + 2 * E + e] + sm[L.part + 3 * E + e]);
        cluster.sync();
        const int eh = E / 2;
        for (int e = rank * eh + tid; e < (rank + 1) * eh; e += AF_THREADS) {
            const float mine = sm[L.ctxp + e], other = peer_sm[L.ctxp + e];
            const float cx = rank == 0 ? mine + other : other + mine;
            if (a.ctx_out) a.ctx_out[(size_t)b * a.ctx_ld + e] = cx;
            if (a.ctx_bf.n) bf_store1(a.ctx_bf, b, e, cx);
        }
    }
    cluster.sync();      // the peer may still be reading this CTA's shared memory
}

// ------------------------------------------------------------------------------------ backward
struct AttnC2BwdSmem {
    int dctx, w, de, v, wld4, wlc, dsb, dconvT, dq, dqp, part, xch, scratch, ths, total;
    __host__ __device__ AttnC2BwdSmem(int N, int E) {
        const AttnC2Geom g(N);
        int o = 0;
        auto take = [&](int n) { int r = o; o += (n + 3) & ~3; return r; };
        dctx = take(E);
        w = take(g.NH);
        de = take(g.NH);
        v = take(AF_D);
        wld4 = take(AF_D * AF_F);
        wlc = take(AF_F * 2 * AF_KS);
        dsb = take(AF_WARPS * 6 * AF_D);          // up to 6 tokens per warp group in the backward dense transpose
        dconvT = take(AF_F * g.NDS);
        dq = take(AF_WARPS * AF_D);
        dqp = take(AF_D);       // this CTA's partial d q, read by rank 0
        part = take(AF_F * 2 * g.NH > 4096 ? AF_F * 2 * g.NH : 4096);      // conv-transpose partials, then [8][A/2] d h_q partials (A <= 1024)
        xch = take(8);
        scratch = take(64);
        ths = take(g.NH * AF_D);    // stashed tanh rows of the own tokens, prefetched with cp.async in the PDL prologue
        total = o;
    }
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(AF_THREADS, 1) k_attention_bwd_c2(const AttnBwdArgs a) {
    extern __shared__ __align__(16) float sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int N = a.s.N, E = a.s.E;
    const AttnC2Geom G(N);
    const AttnC2BwdSmem L(N, E);
    const int rank = (int)cluster.block_rank(), peer = rank ^ 1;
    const int b = blockIdx.x >> 1, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int len = a.lengths ? (int)a.lengths[b] : N;
    const int n_lo = rank * G.NH;
    const int n_own = max(0, min(N, n_lo + G.NH) - n_lo);
    const int own_len = max(0, min(len, n_lo + n_own) - n_lo);     // unmasked own tokens

    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 0] = clock64();
    pdl_trigger();
    {   // the forward pass wrote the tanh stash long ago: asynchronous prefetch of the own tokens' rows
        const float *src = a.th + ((size_t)b * N + n_lo) * AF_D;
        for (int i = tid; i < n_own * (AF_D / 4); i += AF_THREADS) cp_async16(sm + L.ths + i * 4, src + (size_t)i * 4, true);
        cp_async_commit();
    }
    if (tid < AF_D) sm[L.v + tid] = a.v[tid];
    for (int i = tid; i < AF_D * AF_F; i += AF_THREADS) {
        const int d = i >> 5, f = i & 31;
        sm[L.wld4 + ((d >> 2) * AF_F + f) * 4 + (d & 3)] = a.wld[i];
    }
    for (int i = tid; i < AF_F * 2 * AF_KS; i += AF_THREADS) sm[L.wlc + i] = a.wlc[i];
    for (int i = tid; i < AF_F * G.NDS; i += AF_THREADS) sm[L.dconvT + i] = 0.f;
    // forward stash (alignments of this step) and, when they come from the time-batched GEMMs that ran before the chain, the
    // two static d ctx contributions: DRAM-resident, so their latency is taken here, under the previous kernel (E <= 512:
    // one element per thread)
    for (int n = tid; n < G.NH; n += AF_THREADS) sm[L.w + n] = n < n_own ? a.w_t[(size_t)b * a.w_bstride + n_lo + n] : 0.f;
    float x12 = 0.f;
    if (a.dctx12_static && tid < E) {
        x12 = src_get(a.dctx1, b, tid);
        if (a.dctx2.nsplit) x12 += src_get(a.dctx2, b, tid);
    }
    pdl_wait();
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 1] = clock64();
    if (tid < E) {
        const int e = tid;
        float x = x12;
        if (!a.dctx12_static) {
            x = src_get(a.dctx1, b, e);
            if (a.dctx2.nsplit) x += src_get(a.dctx2, b, e);
        }
        if (a.dctx3.nsplit) x += src_get(a.dctx3, b, e);
        sm[L.dctx + e] = x;
        if (rank == 0) a.dctx_out[(size_t)b * E + e] = x;
    }
    cp_async_wait<0>();
    __syncthreads();
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 2] = clock64();

    // ---- d w of the own tokens
    {
        const float *mem_b = a.memory + ((size_t)b * N + n_lo) * E;
        // a warp owns tokens wid, wid + 16, ...; it works on up to 3 of them at a time with every memory / carry load of
        // the batch issued before the first use (the rolled per-token loop paid one L2 round trip + one shuffle tree each)
        constexpr int DWB = 3;
        if (a.memb) {
            // bf16 copy of the encoder memory (written by the fused forward chain): half the L2 traffic of the phase, which is
            // bound by it (19.7 MB of fp32 memory per step over all CTAs = 3100 cycles at the L2 throughput cap)
            const __nv_bfloat16 *memb_b = a.memb + ((size_t)b * N + n_lo) * E;
            constexpr int DWQ = 5;                 // all tokens of the warp at once: 5 x 2 x 16 B per lane
            for (int n0 = wid; n0 < G.NH; n0 += AF_WARPS * DWQ) {
                uint4 mv[DWQ][2];
                float carry[DWQ];
#pragma unroll
                for (int q = 0; q < DWQ; ++q) {
                    const int n = n0 + q * AF_WARPS;
                    const bool live = n < own_len;
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int e = lane * 8 + 256 * i;
                        mv[q][i] = live && e < E ? __ldg(reinterpret_cast<const uint4 *>(memb_b + (size_t)n * E + e)) : make_uint4(0u, 0u, 0u, 0u);
                    }
                    carry[q] = 0.f;
                    if (live) {
                        const size_t gi = (size_t)b * N + n_lo + n;
                        carry[q] = a.dw_carry[gi] + a.dcum_carry[gi];
                        if (a.d_align) carry[q] += a.d_align[(size_t)b * a.da_bstride + n_lo + n];
                    }
                }
                float part[DWQ];
#pragma unroll
                for (int q = 0; q < DWQ; ++q) {
                    part[q] = 0.f;
#pragma unroll
                    for (int i = 0; i < 2; ++i) {
                        const int e = lane * 8 + 256 * i;
                        if (e < E) {
                            const float4 g0 = *reinterpret_cast<const float4 *>(sm + L.dctx + e);
                            const float4 g1 = *reinterpret_cast<const float4 *>(sm + L.dctx + e + 4);
                            const uint4 m = mv[q][i];
                            part[q] = fmaf(__uint_as_float(m.x << 16), g0.x, part[q]); part[q] = fmaf(__uint_as_float(m.x & 0xffff0000u), g0.y, part[q]);
                            part[q] = fmaf(__uint_as_float(m.y << 16), g0.z, part[q]); part[q] = fmaf(__uint_as_float(m.y & 0xffff0000u), g0.w, part[q]);
                            part[q] = fmaf(__uint_as_float(m.z << 16), g1.x, part[q]); part[q] = fmaf(__uint_as_float(m.z & 0xffff0000u), g1.y, part[q]);
                            part[q] = fmaf(__uint_as_float(m.w << 16), g1.z, part[q]); part[q] = fmaf(__uint_as_float(m.w & 0xffff0000u), g1.w, part[q]);
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                    for (int q = 0; q < DWQ; ++q) part[q] += __shfl_xor_sync(0xffffffffu, part[q], o);
                }
#pragma unroll
                for (int q = 0; q < DWQ; ++q) {
                    const int n = n0 + q * AF_WARPS;
                    if (lane == 0 && n < G.NH) sm[L.de + n] = n < own_len ? part[q] + carry[q] : 0.f;
                }
            }
        } else
        for (int n0 = wid; n0 < G.NH; n0 += AF_WARPS * DWB) {
            float4 mv[DWB][4];
            float carry[DWB];
#pragma unroll
            for (int q = 0; q < DWB; ++q) {
                const int n = n0 + q * AF_WARPS;
                const bool live = n < own_len;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int e = lane * 4 + 128 * i;
                    mv[q][i] = live && e < E ? *reinterpret_cast<const float4 *>(mem_b + (size_t)n * E + e) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                carry[q] = 0.f;
                if (live) {
                    const size_t gi = (size_t)b * N + n_lo + n;
                    carry[q] = a.dw_carry[gi] + a.dcum_carry[gi];
                    if (a.d_align) carry[q] += a.d_align[(size_t)b * a.da_bstride + n_lo + n];
                }
            }
            float part[DWB];
#pragma unroll
            for (int q = 0; q < DWB; ++q) {
                part[q] = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int e = lane * 4 + 128 * i;
                    if (e < E) {
                        const float4 g4 = *reinterpret_cast<const float4 *>(sm + L.dctx + e);
                        part[q] = fmaf(mv[q][i].x, g4.x, part[q]); part[q] = fmaf(mv[q][i].y, g4.y, part[q]);
                        part[q] = fmaf(mv[q][i].z, g4.z, part[q]); part[q] = fmaf(mv[q][i].w, g4.w, part[q]);
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int q = 0; q < DWB; ++q) part[q] += __shfl_xor_sync(0xffffffffu, part[q], o);
            }
#pragma unroll
            for (int q = 0; q < DWB; ++q) {
                const int n = n0 + q * AF_WARPS;
                if (lane == 0 && n < G.NH) sm[L.de + n] = n < own_len ? part[q] + carry[q] : 0.f;
            }
        }
    }
    __syncthreads();
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 3] = clock64();
    // ---- softmax backward: <w, dw> over the whole row = rank 0 part + rank 1 part
    const float *peer_sm = cluster.map_shared_rank(sm, peer);
    {
        float part = 0.f;
        for (int n = tid; n < n_own; n += AF_THREADS) part = fmaf(sm[L.w + n], sm[L.de + n], part);
        part = block_sum(part, sm + L.scratch);
        if (tid == 0) sm[L.xch + 0] = part;
        cluster.sync();
        const float other = peer_sm[L.xch + 0];
        const float dot = rank == 0 ? part + other : other + part;
        for (int n = tid; n < G.NH; n += AF_THREADS) {
            const float de = n < n_own ? sm[L.w + n] * (sm[L.de + n] - dot) : 0.f;
            sm[L.de + n] = de;
            if (n < n_own) a.de_out[(size_t)b * N + n_lo + n] = de;
        }
    }
    __syncthreads();
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 4] = clock64();

    // ---- d s, partial d q, d conv of the own tokens
    {
        const float4 v4 = *reinterpret_cast<const float4 *>(sm + L.v + lane * 4);
        float4 dqa = make_float4(0.f, 0.f, 0.f, 0.f);
        // tokens per warp group: as many as it takes for ONE balanced round over the 16 warps (80 own tokens -> 16 groups
        // of 5); with fixed groups of 4 there were 20 groups = two rounds with 12 warps idle in the second
        constexpr int TGM = 6;
        const int tg = min(TGM, max(4, (G.NH + AF_WARPS - 1) / AF_WARPS));
        float *dsb = sm + L.dsb + wid * TGM * AF_D;
        const int ngrp = (G.NH + tg - 1) / tg;
        for (int grp = wid; grp < ngrp; grp += AF_WARPS) {
            const int n0 = grp * tg;
            if (n0 >= own_len) {
                for (int j = 0; j < tg; ++j)
                    if (n0 + j < n_own) a.dconv_out[((size_t)b * N + n_lo + n0 + j) * AF_F + lane] = 0.f;
                continue;
            }
#pragma unroll
            for (int j = 0; j < TGM; ++j) {
                const int n = n0 + j;
                float4 ds = make_float4(0.f, 0.f, 0.f, 0.f);
                if (j < tg && n < own_len) {
                    const float de = sm[L.de + n];
                    const float4 th = *reinterpret_cast<const float4 *>(sm + L.ths + n * AF_D + lane * 4);
                    ds.x = de * v4.x * (1.f - th.x * th.x);
                    ds.y = de * v4.y * (1.f - th.y * th.y);
                    ds.z = de * v4.z * (1.f - th.z * th.z);
                    ds.w = de * v4.w * (1.f - th.w * th.w);
                    dqa.x += ds.x; dqa.y += ds.y; dqa.z += ds.z; dqa.w += ds.w;
                }
                if (j < tg) *reinterpret_cast<float4 *>(dsb + j * AF_D + lane * 4) = ds;
            }
            __syncwarp();
            float acc[TGM];
#pragma unroll
            for (int j = 0; j < TGM; ++j) acc[j] = 0.f;
#pragma unroll 8
            for (int dq = 0; dq < AF_D / 4; ++dq) {
                const float4 w4 = *reinterpret_cast<const float4 *>(sm + L.wld4 + (dq * AF_F + lane) * 4);
#pragma unroll
                for (int j = 0; j < TGM; ++j) {
                    if (j < tg) {
                        const float4 x = *reinterpret_cast<const float4 *>(dsb + j * AF_D + dq * 4);
                        acc[j] = fmaf(x.x, w4.x, fmaf(x.y, w4.y, fmaf(x.z, w4.z, fmaf(x.w, w4.w, acc[j]))));
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < TGM; ++j) {
                const int n = n0 + j;
                if (j < tg && n < n_own) {
                    sm[L.dconvT + lane * G.NDS + n + AF_PAD] = acc[j];       // local index = local token + 15
                    a.dconv_out[((size_t)b * N + n_lo + n) * AF_F + lane] = acc[j];
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
        sm[L.dqp + tid] = q;
    }
    cluster.sync();          // both CTAs' d conv rows and partial d q are complete
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 5] = clock64();
    if (tid < AF_D) {
        const float mine = sm[L.dqp + tid], other = peer_sm[L.dqp + tid];
        const float q = rank == 0 ? mine + other : other + mine;      // always rank 0 + rank 1
        if (rank == 0) {
            if (a.dq_out) a.dq_out[(size_t)b * AF_D + tid] = q;
            if (a.dq_bf.n) bf_store1(a.dq_bf, b, tid, q);
        }
        // operand of the folded query-projection transpose below (rounded to bf16 like the GEMM engine's operands);
        // the per-warp d q partials that lived here are consumed
        if (a.dhq_out) sm[L.dq + tid] = __bfloat162float(__float2bfloat16(q));
    }
    // ---- 15-token halo of d conv from the peer: rank 0 needs the peer's first tokens, rank 1 the peer's last
    for (int i = tid; i < AF_F * AF_PAD; i += AF_THREADS) {
        const int f = i / AF_PAD, h = i - f * AF_PAD;
        if (rank == 0) sm[L.dconvT + f * G.NDS + G.NH + AF_PAD + h] = peer_sm[L.dconvT + f * G.NDS + AF_PAD + h];
        else sm[L.dconvT + f * G.NDS + h] = peer_sm[L.dconvT + f * G.NDS + G.NH + h];
    }
    __syncthreads();
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 6] = clock64();

    // ---- d wcat of the own tokens
    {
        // one task = (filter f, channel c, block of 8 tokens): F * 2 * nblk = 640 tasks keep all 512 threads busy (the
        // first version looped 4 filters per task: 160 tasks, five warps' worth of work on the critical path)
        const int ntask = 2 * G.nblk * AF_F;
        for (int task = tid; task < ntask; task += AF_THREADS) {
            const int f = task & (AF_F - 1), rest = task >> 5;
            const int c = rest / G.nblk, m0 = (rest - c * G.nblk) * 8;
            float acc[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = 0.f;
            {
                float x[40];
                const float4 *xr = reinterpret_cast<const float4 *>(sm + L.dconvT + f * G.NDS + m0);
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
            float4 *dst = reinterpret_cast<float4 *>(sm + L.part + (f * 2 + c) * G.NH + m0);
            dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
            dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
    }
    __syncthreads();
    for (int idx = tid; idx < 2 * n_own; idx += AF_THREADS) {
        const int c = idx / n_own, m = idx - c * n_own;
        float s = 0.f;
#pragma unroll
        for (int f = 0; f < AF_F; ++f) s += sm[L.part + (f * 2 + c) * G.NH + m];
        const size_t gi = (size_t)b * N + n_lo + m;
        if (c == 0) a.dw_carry[gi] = s;
        else a.dcum_carry[gi] += s;
    }
    // ---- d h_att through the query projection (tacotron2.py:98 transposed), folded in here (it used to be a separate K = 128
    // launch of the GEMM engine: two k-blocks on 8 CTAs, ~6 us per step).  Each CTA of the pair takes half of the units:
    // thread = (unit octet tid & 63, d slice tid >> 6 of 16 dims): 16 independent 16-byte loads of the bf16 W_query rows
    // (coalesced along the unit axis) in two batches, then the 8 d slices are summed through shared memory in slice order.
    if (a.dhq_out) {
        __syncthreads();                       // the conv-transpose partials in L.part are consumed
        const int halfA = a.A / 2;             // 512 units per CTA at the default dims
        float *red = sm + L.part;              // [8 d slices][halfA]
        for (int u0 = 0; u0 < halfA; u0 += 512) {
            const int uo = tid & 63, ds = tid >> 6;
            const int u = u0 + 8 * uo;
            float acc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = 0.f;
            if (u < halfA) {
                const __nv_bfloat16 *wp = a.WqB + (size_t)(16 * ds) * a.A + rank * halfA + u;
#pragma unroll
                for (int hb = 0; hb < 2; ++hb) {
                    uint4 wv[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) wv[i] = __ldg(reinterpret_cast<const uint4 *>(wp + (size_t)(8 * hb + i) * a.A));
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const float qv = sm[L.dq + 16 * ds + 8 * hb + i];
                        acc[0] = fmaf(qv, __uint_as_float(wv[i].x << 16), acc[0]); acc[1] = fmaf(qv, __uint_as_float(wv[i].x & 0xffff0000u), acc[1]);
                        acc[2] = fmaf(qv, __uint_as_float(wv[i].y << 16), acc[2]); acc[3] = fmaf(qv, __uint_as_float(wv[i].y & 0xffff0000u), acc[3]);
                        acc[4] = fmaf(qv, __uint_as_float(wv[i].z << 16), acc[4]); acc[5] = fmaf(qv, __uint_as_float(wv[i].z & 0xffff0000u), acc[5]);
                        acc[6] = fmaf(qv, __uint_as_float(wv[i].w << 16), acc[6]); acc[7] = fmaf(qv, __uint_as_float(wv[i].w & 0xffff0000u), acc[7]);
                    }
                }
                float4 *dst = reinterpret_cast<float4 *>(red + ds * halfA + u);
                dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
                dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
            }
            __syncthreads();
            for (int uu = u0 + tid; uu < min(u0 + 512, halfA); uu += AF_THREADS) {
                float v = 0.f;
#pragma unroll
                for (int k = 0; k < 8; ++k) v += red[k * halfA + uu];
                a.dhq_out[(size_t)b * a.A + rank * halfA + uu] = v;
            }
        }
    }
    if (a.dbg && blockIdx.x == 0 && tid == 0 && a.dbg_t < 1024) a.dbg[a.dbg_t * 32 + 7] = clock64();
    cluster.sync();
}

inline bool attention_c2_enabled() {
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("GVX_ATT_C2");
        on = (e && e[0] == '0') ? 0 : 1;
    }
    return on == 1;
}

inline bool attention_fwd_uses_c2(const AttnShape &s) {
    const AttnC2FwdSmem L(s.N, s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    // the split pays when the rows alone cannot fill the machine
    return attention_c2_enabled() && attention_fast_ok(s) && s.B <= 74 && s.N >= 32 && s.E % 8 == 0 && bytes <= 200 * 1024;
}
template <bool WIN>
inline int launch_attention_fwd_c2_k(const AttnFwdArgs &a, size_t bytes, cudaStream_t stream) {
    static size_t configured = 0;      // per instantiation
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_fwd_c2<WIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_fwd_c2<WIN>, dim3(2 * a.s.B), dim3(AF_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    return 0;
}

inline int launch_attention_fwd_best(const AttnFwdArgs &a, cudaStream_t stream) {
    const AttnC2FwdSmem L(a.s.N, a.s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    if (!attention_fwd_uses_c2(a.s)) {
        GVX_CHECK(!a.th_bf16, "the bf16 tanh stash is only written by the cluster attention kernel");
        return launch_attention_fwd_any(a, stream);
    }
    return a.win_fwd ? launch_attention_fwd_c2_k<true>(a, bytes, stream) : launch_attention_fwd_c2_k<false>(a, bytes, stream);
}

inline bool attention_bwd_uses_c2(const AttnShape &s) {
    const AttnC2BwdSmem L(s.N, s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    // (the d w phase of the cluster kernel covers the encoder dim with 4 x 128-wide passes)
    return attention_c2_enabled() && attention_fast_ok(s) && s.B <= 74 && s.N >= 32 && s.E % 8 == 0 && s.E <= 512 && bytes <= 200 * 1024;
}

inline int launch_attention_bwd_best(const AttnBwdArgs &a, cudaStream_t stream) {
    const AttnC2BwdSmem L(a.s.N, a.s.E);
    const size_t bytes = (size_t)L.total * sizeof(float);
    if (!attention_bwd_uses_c2(a.s))
        return launch_attention_bwd_any(a, stream);
    static size_t configured = 0;
    if (bytes > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_attention_bwd_c2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        configured = bytes;
    }
    GVX_CUDA(launch_pdl(k_attention_bwd_c2, dim3(2 * a.s.B), dim3(AF_THREADS), bytes, stream, a));
    GVX_LAUNCHED(1);
    return 0;
}

}  // namespace gvx
