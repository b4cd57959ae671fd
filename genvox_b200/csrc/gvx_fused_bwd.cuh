// genvox_b200 — backward through time of the ATTENTION CHAIN of the decoder in ONE persistent launch (bf16 mode).
//
// The reference has no backward source: `loss["loss"].backward()` (/root/reference/models/tts/tacotron2.py:520) drives
// torch autograd over the T-step graph of Decoder.decode (:333-363).  This kernel is the reverse-time mirror of
// k_att_chain_fwd (gvx_fused_fwd.cuh): for t = T-1 .. 0
//     d ctx_t   = (projection + decoder-LSTM input, both time-batched before the chain) + d x_att_{t+1}[ctx columns]
//     attention backward (:89-129 transposed): d w = <memory, d ctx> + carries, softmax backward -> d e,
//                d s = d e * v * (1 - tanh^2), d q = sum_n d s, d conv = d s . W_loc_dense, conv transpose -> d w / d cum carries
//     d h_att_t = d q . W_query + (decoder-LSTM input) + d x_att_{t+1}[h_att columns]
//     attention-LSTM cell backward -> d gates_t (bf16)
//     d x_att_t[ctx | h_att columns] = d gates_t . W_att[:, ctx | h_att]      (the prenet columns are one time-batched GEMM afterwards)
//
//   * grid = 128 CTAs (one per SM, all co-resident) in 32 clusters of 4.
//   * the recurrent GEMM (K = 4A = 4096 gate rows, 1536 output columns) is split like k_lstm_chain_bwd: cluster c owns 48
//     output columns (h_att units 32c..32c+31 and ctx columns 16c..16c+15), CTA rank r of the cluster contracts K quarter r
//     with its [48 x 1024] bf16 slice of W_att^T resident in shared memory for the whole sequence (96 KB, SWIZZLE_128B).
//     Per step the K quarter of the d-gates image ([64 rows x 1024] bf16, written by 32 CTAs) is streamed by TMA bulk
//     copies through a 4-slot ring into tcgen05.mma (UMMA 64 x 48 x 16, accumulator in TMEM); the four fp32 partial tiles are
//     exchanged through distributed shared memory and summed in rank order (deterministic).  Rank r finishes the h_att
//     columns of ITS OWN 8 hidden units (they never leave the CTA: thread = (batch row, unit) keeps d c and the recurrent
//     part of d h in registers) and 4 ctx columns, which it publishes as (value, step tag) 64-bit words.
//   * the attention backward is row-parallel: RS = 2 (B <= 64) or 4 (B <= 32) CTAs of one cluster share a batch row
//     (token ranges); <w, d w>, d q and a 15-token halo of d conv are exchanged through distributed shared memory with
//     mbarrier arrive/wait pairs.  The d w / d cum carries of the own tokens live in shared memory for the whole sequence.
//     The tanh stash of the own tokens (bf16, chunk-swizzled by the forward kernel) is prefetched one step ahead by a TMA
//     bulk copy; the bf16 encoder-memory rows of the d w phase are requested before the step's d ctx has arrived.
//     d conv = d s . W_loc_dense runs on mma.sync with a 3-pass bf16 split (hi*hi + lo*hi + hi*lo: fp32-grade accuracy).
//   * exchanges between the two decompositions carry their own readiness: d q rows and d ctx columns travel as
//     (value, tag) words the consumers poll; the only counter barrier per step guards the d-gates image (TMA cannot poll),
//     one counter per K quarter (32 arrivals).
//
// Every wait is bounded (fa_spin): on timeout an error code is recorded, the grid drains and the host raises.
#pragma once
#include <cooperative_groups.h>
#include <cuda_bf16.h>

#include "gvx_fused_fwd.cuh"

namespace gvx {

constexpr int FB_THREADS = 512;
constexpr int FB_NCOL = 48;                        // output columns per cluster: 32 h_att units + 16 ctx columns
constexpr int FB_KSLAB = 16;                       // 64-row K slabs of one K quarter (A = 1024)
constexpr int FB_WSLAB_BYTES = FB_NCOL * 128;      // one K slab of the resident weight slice
constexpr int FB_RING = 8;                         // slots 0..3 dedicated, 4..7 alias buffers only the attention phase uses
constexpr int FB_WLD_LD = 136;                     // bf16 per row of the W_loc_dense^T tile (conflict-free B fragments)
constexpr int FB_QBYTES = FB_KSLAB * PC_CHUNK_BYTES;   // one K quarter of the d-gates image
constexpr int FB_PLD = 68;                         // row stride of a partial-tile column: pushes stay contiguous, the (row, unit) reads conflict-free
constexpr int FB_DWQ = 5;                          // tokens per warp whose memory rows are requested a phase ahead

struct FbGeom {
    int RS, NH, NHP, nblk, NDS, nmt;
    __host__ __device__ FbGeom(int N, int RS_) {
        RS = RS_;
        NH = (((N + RS - 1) / RS) + 7) & ~7;       // tokens per CTA
        NHP = (NH + 15) & ~15;                     // rounded to mma row tiles
        nblk = NH / 8;
        NDS = NH + 40;                             // local d conv row: 15-token halo on both sides
        nmt = NHP / 16;
    }
};

struct FbShared {
    uint64_t full[FB_RING], empty[FB_RING], tmem_full, wbar, thbar, xb[4];     // xb: [0] carry dots, [1] gathered d q rows, [2] d conv halos, [3] partial tiles
    uint32_t tmem_slot;
    volatile int dead;
};

struct FbSmem {      // byte offsets from the 1 KB aligned base
    int ring, ths, dhqp, dqs, pdw, wsm, pin, cpart, dconvT, wlc, wldh, dctx, ctx32, w, de, dal, dwc, dcumc, v, xch, sh, total;
    __host__ __device__ FbSmem(int N, int RS) {
        const FbGeom g(N, RS);
        int o = 0;
        auto take = [&](int bytes) { int r = o; o += (bytes + 127) & ~127; return r; };
        // The TMA ring of the d-gates image (8 slots, in use between the image barrier and the end of the GEMM) is time-shared
        // with everything only the attention / cell phases of a step touch:
        //   tanh -> d s tile (lands before the step, dead after the d conv contraction), the gathered d q rows and the d h_q
        //   partials of the cell phase, the per-warp d w partials.
        ring = 0;
        ths = take(g.NHP * AF_D * 2);
        dqs = take(PC_ROWS * AF_D * 2);                       // [64 rows][128] bf16 d q of all rows (chunk-swizzled), pushed by the 4 ranks
        dhqp = take(4 * PC_ROWS * 8 * 4);                     // [4 k quarters][64 rows][8 units]
        pdw = take(16 * g.NHP * 4);                           // [16 warps][tokens] d w partials
        o = o > FB_RING * PC_CHUNK_BYTES ? ((o + 1023) & ~1023) : FB_RING * PC_CHUNK_BYTES;
        wsm = take(FB_KSLAB * FB_WSLAB_BYTES);
        pin = take(4 * 12 * FB_PLD * 4);                      // partial tiles pushed by the 4 ranks: [src rank][8 h_att + 4 ctx columns][68: 64 rows + pad]
        cpart = take(16 * 2 * g.NHP * 4);                     // conv-transpose partials
        dconvT = take(AF_F * g.NDS * 4);
        wlc = take(AF_F * 2 * AF_KS * 4);
        wldh = take(AF_F * FB_WLD_LD * 2);
        dctx = take(FA_E * 4);
        ctx32 = take(FA_E * 4);
        w = take(g.NHP * 4);
        de = take(g.NHP * 4);
        dal = take(g.NHP * 4);
        dwc = take(g.NHP * 4);
        dcumc = take(g.NHP * 4);
        v = take(AF_D * 4);
        xch = take(64);                                       // [0..3] carry dots pushed by the parts of the row
        sh = take((int)sizeof(FbShared));
        total = o + 1024;
    }
};

struct FbArgs {
    const __nv_bfloat16 *Wimg;       // [128 CTAs][16 slabs][48 rows][128 B] SWIZZLE_128B (k_fb_pack_w)
    uint8_t *gimg;                   // [2][4 K quarters][16 slabs][64 rows][128 B] d-gates image, zero at launch
    const __nv_bfloat16 *WqB;        // [D][A] row-major bf16
    const float *gates_stash;        // [T][B][4A]
    const float *c_stash;            // [T+1][B][A]
    const float *dxdall;             // [T][B][A+E]: d [h_att | ctx] from the decoder-LSTM input
    const float *dhc;                // [T][B][Kp]: d [h_dec | ctx] from the projections (ctx at column H)
    int Kp, H;
    const float *d_align;            // [B][T][N] or null
    const float *align;              // [B][T][N]
    const float *ctx32;              // [T][B][E] fp32 attention context of the forward pass
    const __nv_bfloat16 *th;         // [T][B][N][D] bf16, 16-byte chunks swizzled by (token & 7)
    const __nv_bfloat16 *memb;       // [B][N][E]
    const float *wlc, *wldT, *v;     // location conv [F][2][KS], location dense transposed [F][D], v [D]
    const int64_t *lengths;
    __nv_bfloat16 *dg_rm;            // [T][B][4A]
    __nv_bfloat16 *dq_rm;            // [T][B][D]
    float *de_out;                   // [T][B][N]
    uint16_t *dconv_out;             // [T][B][N][F] bf16: the A operand of k_post_conv_stream (gvx_post_tc.cuh)
    float *dctx_out;                 // [T][B][E]
    unsigned long long *dctxx;       // [2][64][E]   (value, tag) exchange of the recurrent d ctx part, zero at launch
    unsigned long long *dqx;         // [2][64][4 parts][D/2] (bf16x2, tag) exchange of the per-part d q, zero at launch
    unsigned *bar;                   // [4 K quarters][16 slabs] counters (one 64-byte line per quarter, zero at launch): the two CTAs
                                     // that own the 16 hidden units of a 64-row K slab of the d-gates image have written it
    int *err;
    DropCfg drop;
    int row_offset, B, N, T, RS;
    long long *dbg;
};

__device__ __forceinline__ void fb_gstamp(long long *dbg, int cta, int i, int k) {
    if (dbg && i == 20) dbg[32 * 1024 + cta * 16 + k] = fa_globaltimer();
}
__device__ __forceinline__ void fb_bar_w14() { asm volatile("bar.sync 2, 448;" ::: "memory"); }
// Push into another CTA's shared memory with the arrival folded into the store: the 4 / 8 bytes are counted on the
// receiver's mbarrier (complete_tx), which the receiver arms with the byte count of the phase (expect_tx).  No fence on
// either side (a release-arrive at cluster scope compiles to MEMBAR.ALL.GPU: it waits for every global store in flight).
__device__ __forceinline__ void st_async_f32(uint32_t caddr, float v, uint32_t cmbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.f32 [%0], %1, [%2];" ::"r"(caddr), "f"(v), "r"(cmbar) : "memory");
}
__device__ __forceinline__ void st_async_f32x2(uint32_t caddr, float v0, float v1, uint32_t cmbar) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.f32 [%0], {%1, %2}, [%3];" ::"r"(caddr), "f"(v0), "f"(v1), "r"(cmbar)
                 : "memory");
}
// mbarrier wait of a whole warp: ONE lane polls (hundreds of threads spinning on mbarriers that share a shared-memory line
// with the TMA ring's full / empty barriers slow the single-thread TMA and MMA loops down), the result is broadcast
__device__ __forceinline__ bool fb_wait_warp(uint64_t *bar, uint32_t parity, volatile int *dead, int *err, int code) {
    int ok = 1;
    if ((threadIdx.x & 31) == 0) ok = fa_wait_cluster(bar, parity, dead, err, code) ? 1 : 0;
    ok = __shfl_sync(0xffffffffu, ok, 0);
    // Every lane then performs its OWN acquire on the (already completed) phase: data written by st.async pushes / TMA is only
    // guaranteed visible to threads that have observed the barrier themselves - a lane that merely learns of the completion
    // through a shuffle read stale shared memory in the forward chain (seen as run-dependent wrong results).
    if (ok) {
        while (!mbar_try_wait_cluster(bar, parity)) {}
    }
    return ok != 0;
}
// lstm_bwd_point (gvx_gemm.cuh) with the SFU tanh the fused forward chain used for h = o * tanh(c)
__device__ __forceinline__ float4 fb_lstm_bwd_point(float dh_dropped, float mult, float4 ga, float c_prev, float c_new, float dc_in,
                                                    float &dc_prev) {
    const float dh = dh_dropped * mult;
    const float tc = tanh_fast(c_new);
    const float d_o = dh * tc;
    const float dc = dc_in + dh * ga.w * (1.f - tc * tc);
    const float d_i = dc * ga.z, d_g = dc * ga.x, d_f = dc * c_prev;
    dc_prev = dc * ga.y;
    return make_float4(d_i * ga.x * (1.f - ga.x), d_f * ga.y * (1.f - ga.y), d_g * (1.f - ga.z * ga.z), d_o * ga.w * (1.f - ga.w));
}

__global__ void __cluster_dims__(4, 1, 1) __launch_bounds__(FB_THREADS, 1) k_att_chain_bwd(const FbArgs a) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const int N = a.N, T = a.T, B = a.B, RS = a.RS;
    const FbGeom G(N, RS);
    const FbSmem L(N, RS);
    uint8_t *ring = smem + L.ring, *wsm = smem + L.wsm, *ths = smem + L.ths;
    float *pin = (float *)(smem + L.pin), *cpart = (float *)(smem + L.cpart), *pdw = (float *)(smem + L.pdw);
    uint8_t *dqs = smem + L.dqs;
    float *dconvT = (float *)(smem + L.dconvT), *wlc = (float *)(smem + L.wlc);
    __nv_bfloat16 *wldh = (__nv_bfloat16 *)(smem + L.wldh);
    float *dctx = (float *)(smem + L.dctx), *ctx32 = (float *)(smem + L.ctx32);
    float *ws = (float *)(smem + L.w), *des = (float *)(smem + L.de), *dals = (float *)(smem + L.dal);
    float *dwc = (float *)(smem + L.dwc), *dcumc = (float *)(smem + L.dcumc), *vs = (float *)(smem + L.v);
    float *dhqp = (float *)(smem + L.dhqp);
    float *xch = (float *)(smem + L.xch);
    FbShared *sh = (FbShared *)(smem + L.sh);

    const int tid = threadIdx.x, wid = tid >> 5, lane = tid & 31, j = blockIdx.x;
    const int g4 = lane >> 2, tig = lane & 3;
    const int r = (int)cluster.block_rank(), c = j >> 2;            // r == j & 3
    const int row = RS == 2 ? 2 * c + (r >> 1) : c;
    const int prt = RS == 2 ? (r & 1) : r;                          // which token range of the row
    const int gbase = RS == 2 ? (r & ~1) : 0;                       // cluster rank of part 0 of this row
    const bool rvalid = row < B;
    const int rowc = rvalid ? row : B - 1;
    const int len = a.lengths ? (int)a.lengths[rowc] : N;
    const int n_lo = prt * G.NH;
    const int n_own = rvalid ? max(0, min(N, n_lo + G.NH) - n_lo) : 0;
    const int own_len = max(0, min(len, n_lo + n_own) - n_lo);
    const bool th_live = n_own > 0;
    const bool has_left = prt > 0, has_right = prt < RS - 1;
    // unit side: thread = (batch row ub, hidden unit 8j + uk), unit fastest: 8 consecutive lanes read / write one contiguous run of
    // a row of the gate stash, the d-gates image and the row-major d gates (with the row fastest every warp-level access
    // touched 32 different lines: ~1500 cycles of LSU time per step)
    const int uk = tid & 7, ub = tid >> 3, uu = 8 * j + uk;
    const int ck = tid & 3, cb = (tid >> 2) & 63;                  // ctx-column side of the GEMM epilogue (threads 0..255)
    const bool uvalid = ub < B;

    if (tid == 0) {
        for (int s = 0; s < FB_RING; ++s) { mbar_init(sh->full + s, 1); mbar_init(sh->empty + s, 1); }
        mbar_init(&sh->tmem_full, 1);
        mbar_init(&sh->wbar, 1);
        mbar_init(&sh->thbar, 1);
        // exchange barriers: one local arrive.expect_tx per phase, the remote st.async pushes complete the byte count
        for (int k = 0; k < 4; ++k) mbar_init(sh->xb + k, 1);
        sh->dead = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (wid == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_slot)), "n"(64) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (int i = tid; i < AF_F * 2 * AF_KS; i += FB_THREADS) wlc[i] = a.wlc[i];
    for (int i = tid; i < AF_F * AF_D; i += FB_THREADS) wldh[(i >> 7) * FB_WLD_LD + (i & 127)] = __float2bfloat16(a.wldT[i]);   // [f][d]
    if (tid < AF_D) vs[tid] = a.v[tid];
    for (int i = tid; i < AF_F * G.NDS; i += FB_THREADS) dconvT[i] = 0.f;
    for (int i = tid; i < G.NHP * AF_D / 2; i += FB_THREADS) reinterpret_cast<uint32_t *>(ths)[i] = 0u;
    for (int i = tid; i < G.NHP; i += FB_THREADS) { ws[i] = 0.f; des[i] = 0.f; dals[i] = 0.f; dwc[i] = 0.f; dcumc[i] = 0.f; }
    if (tid < 16) xch[tid] = 0.f;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh->tmem_slot;
    if (tid == 0) {
        // resident weight slice; first tanh tile (the zero fill above went through the generic proxy)
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(&sh->wbar, FB_KSLAB * FB_WSLAB_BYTES);
        const uint8_t *wsrc = (const uint8_t *)a.Wimg + (size_t)j * FB_KSLAB * FB_WSLAB_BYTES;
        for (uint32_t off = 0; off < FB_KSLAB * FB_WSLAB_BYTES; off += 16384) tma_bulk_g2s(wsm + off, wsrc + off, 16384, &sh->wbar);
        if (th_live) {
            mbar_expect_tx(&sh->thbar, (uint32_t)n_own * AF_D * 2);
            tma_bulk_g2s(ths, a.th + (((size_t)(T - 1) * B + row) * N + n_lo) * AF_D, (uint32_t)n_own * AF_D * 2, &sh->thbar);
        }
    }
    // W_query^T fragments of the own 8 units: warp (m tile = wid & 3, k quarter = wid >> 2) contracts d in [32 kq, 32 kq + 32)
    const int qm = wid & 3, kq = wid >> 2;
    uint32_t wqf[2][2];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
            const int d0 = 16 * (2 * kq + s) + 2 * tig + 8 * hh;
            const __nv_bfloat16 lo = a.WqB[(size_t)d0 * FA_A + 8 * j + g4], hi = a.WqB[(size_t)(d0 + 1) * FA_A + 8 * j + g4];
            wqf[s][hh] = (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
        }
    // DSMEM addresses
    const uint32_t my_xch = smem_u32(xch), my_xb0 = smem_u32(sh->xb + 0), my_xb3 = smem_u32(sh->xb + 3), my_pin = smem_u32(pin);
    const uint32_t halo_bytes = (uint32_t)(min(AF_PAD, G.NH) * AF_F * 4) * (uint32_t)((has_left ? 1 : 0) + (has_right ? 1 : 0));
    const uint32_t my_dqs = smem_u32(dqs), my_xb1 = smem_u32(sh->xb + 1);
    const uint32_t nbl_dconv = mapa_u32(smem_u32(dconvT), (uint32_t)(gbase + max(prt - 1, 0)));
    const uint32_t nbr_dconv = mapa_u32(smem_u32(dconvT), (uint32_t)(gbase + min(prt + 1, RS - 1)));
    const uint32_t nbl_xb2 = mapa_u32(smem_u32(sh->xb + 2), (uint32_t)(gbase + max(prt - 1, 0)));
    const uint32_t nbr_xb2 = mapa_u32(smem_u32(sh->xb + 2), (uint32_t)(gbase + min(prt + 1, RS - 1)));

    // dropout stream: the seed words are read from device memory ONCE (a load per step sat in front of the Philox rounds)
    DropCfg drop = a.drop;
    if (drop.kptr) { drop.k0 = drop.kptr[0]; drop.k1 = drop.kptr[1]; drop.kptr = nullptr; }
    // carried per thread on the unit side
    float dc = 0.f, rec = 0.f;
    float c_new = uvalid ? a.c_stash[((size_t)T * B + ub) * FA_A + uu] : 0.f;
    const int quarter = j >> 5;                                  // K quarter the own d gates belong to
    const int kk0 = 4 * uu - 1024 * quarter;                     // k inside the quarter of gate row 4 * uu
    const size_t gimg_off = (size_t)quarter * FB_QBYTES + (size_t)(kk0 >> 6) * PC_CHUNK_BYTES + ub * 128 +
                            ((((kk0 & 63) >> 3) ^ (ub & 7)) << 4) + (kk0 & 7) * 2;
    unsigned *bq_own = a.bar + 16 * quarter + ((j & 31) >> 1);      // slab of the image the own 8 units belong to
    const unsigned *bq_need = a.bar + 16 * r;                      // the 16 slab counters of the K quarter this CTA contracts
    const size_t AE = FA_A + FA_E;

    // static inputs of the first attention step
    if (tid < FA_E) {
        dctx[tid] = rvalid ? a.dhc[((size_t)(T - 1) * B + row) * a.Kp + a.H + tid] + a.dxdall[((size_t)(T - 1) * B + row) * AE + FA_A + tid] : 0.f;
        ctx32[tid] = rvalid ? a.ctx32[((size_t)(T - 1) * B + row) * FA_E + tid] : 0.f;
    }
    if (tid < G.NHP) {
        ws[tid] = tid < n_own ? a.align[((size_t)row * T + (T - 1)) * N + n_lo + tid] : 0.f;
        dals[tid] = (a.d_align && tid < n_own) ? a.d_align[((size_t)row * T + (T - 1)) * N + n_lo + tid] : 0.f;
    }
    if (wid == 0 && a.d_align && rvalid) {
        // carry dots of the first step: <w_{T-1}, d align_{T-1}> of every part of the row (there are no carries yet, but the
        // alignment gradient is part of d w).  Later steps get theirs pushed by the parts; this sums in the same order as the
        // parts do, so a run is bit-identical to the prefix of a longer run whose upstream gradient is zero after it.
        const float *al = a.align + ((size_t)row * T + (T - 1)) * N, *dal = a.d_align + ((size_t)row * T + (T - 1)) * N;
        for (int q = 0; q < RS; ++q) {
            const int q_lo = q * G.NH, q_own = max(0, min(N, q_lo + G.NH) - q_lo), q_len = max(0, min(len, q_lo + q_own) - q_lo);
            float p = 0.f;
            for (int n = lane; n < q_len; n += 32) p = fmaf(al[q_lo + n], dal[q_lo + n], p);
            p = warp_sum(p);
            if (lane == 0) xch[q] = p;
        }
    }
    __syncthreads();
    cluster.sync();          // every CTA's mbarriers are initialised before any remote arrive
    const bool okw = fa_wait_mbar(&sh->wbar, 0, &sh->dead, a.err, 51);

    // dropout multiplier of (row ub, unit uu) at the step about to be processed: computed a phase ahead (Philox: ~100 instructions)
    float mult = uvalid ? drop_mult(drop, SITE_ATT, (uint32_t)(T - 1), (uint32_t)(ub + a.row_offset), (uint32_t)uu) : 1.f;
    const __nv_bfloat16 *memb_b = a.memb + ((size_t)rowc * N + n_lo) * FA_E;
    // bf16 encoder-memory operand of the d w contraction, in mma.sync A-fragment layout: warp w owns encoder columns
    // [32 w, 32 w + 32) for ALL tokens, lane (g4, tig) holds 8 consecutive columns of tokens 16 mt + g4 and 16 mt + g4 + 8.
    // The first FB_DWQ token tiles are always requested a phase ahead of their use.
    uint4 mv[FB_DWQ][2];
    auto load_mem = [&](int mt0) {
#pragma unroll
        for (int q = 0; q < FB_DWQ; ++q) {
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const int n = 16 * (mt0 + q) + g4 + 8 * h2;
                mv[q][h2] = n < own_len ? __ldg(reinterpret_cast<const uint4 *>(memb_b + (size_t)n * FA_E + 32 * wid + 8 * tig)) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
    };
    load_mem(0);
    for (int i = 0; i < T; ++i) {
        const int t = T - 1 - i;
        const uint32_t par = (uint32_t)i & 1u;
        if (tid == 0) { pc_stamp(a.dbg, j, i, 0); fb_gstamp(a.dbg, j, i, 0); }
        // ============================================================ attention backward of step t: the critical path is local
        if (i > 0 && tid < FA_E) {
            // (CTAs without a batch row poll a valid row too: seeing the tags of ALL CTAs is what orders the reuse of buffers)
            const unsigned long long *src = a.dctxx + ((size_t)par * PC_ROWS + rowc) * FA_E + tid;
            unsigned long long wv = 0ull;
            fa_spin([&] { wv = ld_relaxed_u64(src); return (unsigned)(wv >> 32) == (unsigned)i; }, &sh->dead, a.err, 52);
            if (rvalid) dctx[tid] += __uint_as_float((unsigned)wv);
        }
        if (tid < FA_E && rvalid && prt == 0) a.dctx_out[((size_t)t * B + row) * FA_E + tid] = dctx[tid];
        if (i > 0) fb_wait_warp(sh->xb + 0, par ^ 1u, &sh->dead, a.err, 53);         // carry dots of every part (pushed a phase ago)
        if (th_live) fb_wait_warp(&sh->thbar, par, &sh->dead, a.err, 54);
        __syncthreads();
        if (tid == 0) {
            pc_stamp(a.dbg, j, i, 1);
            fb_gstamp(a.dbg, j, i, 1);
            // arm this iteration's exchange phases (the pushes may already be on their way: the byte count is signed)
            mbar_expect_tx(sh->xb + 1, (uint32_t)PC_ROWS * AF_D * 2);
            if (halo_bytes) mbar_expect_tx(sh->xb + 2, halo_bytes);
            if (i + 1 < T) {
                mbar_expect_tx(sh->xb + 0, (uint32_t)RS * 4);
                mbar_expect_tx(sh->xb + 3, 4u * 12u * PC_ROWS * 4u);      // 4 ranks x 12 columns x 64 rows x 4 B
            }
        }
        {   // d w of the own tokens on mma.sync: [tokens x 32 encoder columns of this warp] . [d ctx hi | d ctx lo] (bf16 split of the
            // fp32 d ctx: the bf16 memory operand is exact, so the products carry ~16 mantissa bits), partial per warp
            uint32_t bfr[4] = {0u, 0u, 0u, 0u};
            if (g4 < 2) {
                const float4 d0 = *reinterpret_cast<const float4 *>(dctx + 32 * wid + 8 * tig), d1 = *reinterpret_cast<const float4 *>(dctx + 32 * wid + 8 * tig + 4);
                float x[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
                if (g4 == 1) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) x[k] -= __bfloat162float(__float2bfloat16(x[k]));
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) bfr[k] = pack_bf2(x[2 * k], x[2 * k + 1]);
            }
            for (int mt0 = 0; mt0 < G.nmt; mt0 += FB_DWQ) {
                if (mt0 > 0) load_mem(mt0);
#pragma unroll
                for (int q = 0; q < FB_DWQ; ++q) {
                    if (mt0 + q < G.nmt) {
                        float acc[4] = {0.f, 0.f, 0.f, 0.f};
                        mma_bf16_16816(acc, mv[q][0].x, mv[q][1].x, mv[q][0].y, mv[q][1].y, bfr[0], bfr[1]);
                        mma_bf16_16816(acc, mv[q][0].z, mv[q][1].z, mv[q][0].w, mv[q][1].w, bfr[2], bfr[3]);
                        if (tig == 0) {
                            pdw[wid * G.NHP + 16 * (mt0 + q) + g4] = acc[0] + acc[1];
                            pdw[wid * G.NHP + 16 * (mt0 + q) + g4 + 8] = acc[2] + acc[3];
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) pc_stamp(a.dbg, j, i, 12);
        if (wid * 32 < G.NHP) {   // softmax backward: <w, d w> = <ctx_t, d ctx> + sum over parts <w, carries>  (ctx_t = sum_n w_n memory_n:
            // no exchange with the other token ranges on the critical path)
            float dot = 0.f;
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                const float4 g0 = *reinterpret_cast<const float4 *>(dctx + lane * 8 + 256 * h2), g1 = *reinterpret_cast<const float4 *>(dctx + lane * 8 + 256 * h2 + 4);
                const float4 c0 = *reinterpret_cast<const float4 *>(ctx32 + lane * 8 + 256 * h2), c1 = *reinterpret_cast<const float4 *>(ctx32 + lane * 8 + 256 * h2 + 4);
                dot = fmaf(c0.x, g0.x, dot); dot = fmaf(c0.y, g0.y, dot); dot = fmaf(c0.z, g0.z, dot); dot = fmaf(c0.w, g0.w, dot);
                dot = fmaf(c1.x, g1.x, dot); dot = fmaf(c1.y, g1.y, dot); dot = fmaf(c1.z, g1.z, dot); dot = fmaf(c1.w, g1.w, dot);
            }
            dot = warp_sum(dot);
            for (int p = 0; p < RS; ++p) dot += xch[p];
            const int n = tid;
            if (n < G.NHP) {
                float dwn = 0.f;
#pragma unroll
                for (int w8 = 0; w8 < 16; ++w8) dwn += pdw[w8 * G.NHP + n];
                dwn += (dwc[n] + dcumc[n]) + dals[n];
                const float de = n < own_len ? ws[n] * (dwn - dot) : 0.f;
                des[n] = de;
                if (n < n_own) a.de_out[((size_t)t * B + row) * N + n_lo + n] = de;
            }
        }
        __syncthreads();
        if (tid == 0) pc_stamp(a.dbg, j, i, 13);
        {   // d s = d e * v * (1 - tanh^2) replaces the tanh values in the tile (bf16, same swizzle): it is the A operand of the
            // d conv contraction below.  Warp w owns attention dims [8 w, 8 w + 8) of ALL tokens (lane = token), so its column
            // sums - this part's d q, taken in fp32 before the rounding - need no cross-warp reduction: they are published at once.
            const float4 va = *reinterpret_cast<const float4 *>(vs + 8 * wid), vb = *reinterpret_cast<const float4 *>(vs + 8 * wid + 4);
            const float vv[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
            float acc[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] = 0.f;
            for (int n = lane; n < G.NHP; n += 32) {
                uint4 *tp = reinterpret_cast<uint4 *>(ths + n * 256 + ((wid ^ (n & 7)) << 4));
                const float de = des[n];
                const uint4 tw = *tp;
                const float th[8] = {bf_lo(tw.x), bf_hi(tw.x), bf_lo(tw.y), bf_hi(tw.y), bf_lo(tw.z), bf_hi(tw.z), bf_lo(tw.w), bf_hi(tw.w)};
                float sv[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    sv[k] = n < own_len ? de * vv[k] * (1.f - th[k] * th[k]) : 0.f;
                    acc[k] += sv[k];
                }
                *tp = make_uint4(pack_bf2(sv[0], sv[1]), pack_bf2(sv[2], sv[3]), pack_bf2(sv[4], sv[5]), pack_bf2(sv[6], sv[7]));
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
            }
            if (lane < 4) {
                const float q0 = lane == 0 ? acc[0] : (lane == 1 ? acc[2] : (lane == 2 ? acc[4] : acc[6]));
                const float q1 = lane == 0 ? acc[1] : (lane == 1 ? acc[3] : (lane == 2 ? acc[5] : acc[7]));
                const int d2 = 4 * wid + lane;          // dim pair
                if (rvalid)
                    st_relaxed_u64(a.dqx + (((size_t)par * PC_ROWS + row) * 4 + prt) * (AF_D / 2) + d2,
                                   ((unsigned long long)(unsigned)(i + 1) << 32) | pack_bf2(q0, q1));
            }
        }
        if (tid == 0) { pc_stamp(a.dbg, j, i, 2); fb_gstamp(a.dbg, j, i, 2); }
        // ---- static inputs of the cell backward (unit side): requested now, used after the d q rows have arrived
        float4 ga = make_float4(0.f, 0.f, 0.f, 0.f);
        float c_prev = 0.f, dxd = 0.f;
        if (uvalid) {
            ga = __ldcs(reinterpret_cast<const float4 *>(a.gates_stash + ((size_t)t * B + ub) * 4 * FA_A + 4 * uu));
            c_prev = __ldcs(a.c_stash + ((size_t)t * B + ub) * FA_A + uu);
            dxd = __ldcs(a.dxdall + ((size_t)t * B + ub) * AE + uu);
        }
        if (tid == 0) pc_stamp(a.dbg, j, i, 14);
        // ---- d conv = d s . W_loc_dense on mma.sync (bf16 operands, fp32 accumulate): task = (16-token tile, 16 filters)
        for (int task = wid; task < 2 * G.nmt; task += 16) {
            const int mt = task >> 1, nh = task & 1;
            const int n0 = 16 * mt + g4, n1 = n0 + 8;
            const uint8_t *tr0 = ths + n0 * 256 + 4 * tig, *tr1 = ths + n1 * 256 + 4 * tig;
            const int sw0 = n0 & 7, sw1 = n1 & 7;
            float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
            const __nv_bfloat16 *bh = wldh + (16 * nh + g4) * FB_WLD_LD + 2 * tig;
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                const int ch = 2 * s;                      // 16-byte chunk of d0 = 16 s (+ 8 -> chunk + 1)
                const uint32_t a0 = *reinterpret_cast<const uint32_t *>(tr0 + ((ch ^ sw0) << 4));
                const uint32_t a1 = *reinterpret_cast<const uint32_t *>(tr1 + ((ch ^ sw1) << 4));
                const uint32_t a2 = *reinterpret_cast<const uint32_t *>(tr0 + (((ch + 1) ^ sw0) << 4));
                const uint32_t a3 = *reinterpret_cast<const uint32_t *>(tr1 + (((ch + 1) ^ sw1) << 4));
#pragma unroll
                for (int nt = 0; nt < 2; ++nt) {
                    const uint32_t b0 = *reinterpret_cast<const uint32_t *>(bh + 8 * nt * FB_WLD_LD + 16 * s);
                    const uint32_t b1 = *reinterpret_cast<const uint32_t *>(bh + 8 * nt * FB_WLD_LD + 16 * s + 8);
                    mma_bf16_16816(acc[nt], a0, a1, a2, a3, b0, b1);
                }
            }
#pragma unroll
            for (int nt = 0; nt < 2; ++nt) {
                const int f0 = 16 * nh + 8 * nt + 2 * tig;
#pragma unroll
                for (int hr = 0; hr < 2; ++hr) {
                    const int n = hr == 0 ? n0 : n1;
                    const float x0 = acc[nt][2 * hr], x1 = acc[nt][2 * hr + 1];
                    if (n < G.NH) {
                        dconvT[f0 * G.NDS + AF_PAD + n] = x0;
                        dconvT[(f0 + 1) * G.NDS + AF_PAD + n] = x1;
                        if (n < n_own) *reinterpret_cast<uint32_t *>(a.dconv_out + (((size_t)t * B + row) * N + n_lo + n) * AF_F + f0) = pack_bf2(x0, x1);
                        // 15-token halos pushed straight into the neighbours' windows
                        if (has_left && n < AF_PAD) {
                            st_async_f32(nbl_dconv + 4 * (f0 * G.NDS + AF_PAD + G.NH + n), x0, nbl_xb2);
                            st_async_f32(nbl_dconv + 4 * ((f0 + 1) * G.NDS + AF_PAD + G.NH + n), x1, nbl_xb2);
                        }
                        if (has_right && n >= G.NH - AF_PAD) {
                            st_async_f32(nbr_dconv + 4 * (f0 * G.NDS + n - (G.NH - AF_PAD)), x0, nbr_xb2);
                            st_async_f32(nbr_dconv + 4 * ((f0 + 1) * G.NDS + n - (G.NH - AF_PAD)), x1, nbr_xb2);
                        }
                    }
                }
            }
        }
        if (tid == 0) pc_stamp(a.dbg, j, i, 15);
        __syncthreads();
        if (tid == 0) { pc_stamp(a.dbg, j, i, 3); fb_gstamp(a.dbg, j, i, 3); }

        // ============================================================ attention-LSTM cell backward of step t (unit side)
        {   // d q of all rows.  The per-part rows arrive as (bf16x2, tag) words in global memory; every CTA needs all of them, but the
            // four CTAs of a cluster share the work: rank r polls and reads rows [16 r, 16 r + 16) only (both parts), adds the parts and
            // pushes the bf16 rows into the shared memory of all four ranks (st.async).  A quarter of the L2 / LSU traffic of every
            // CTA reading everything, and the row-major d q stash of the time-batched query-layer gradient falls out of it.
            const int grow = 16 * r + (tid >> 5);
            const unsigned long long *qsrc = a.dqx + ((size_t)par * PC_ROWS + grow) * 4 * (AF_D / 2) + 2 * lane;
            float q4[4] = {0.f, 0.f, 0.f, 0.f};
            if (grow < B) {
                unsigned long long wv[4][2];
                fa_spin([&] {
                    bool all = true;
#pragma unroll
                    for (int p = 0; p < 4; ++p) {
                        if (p < RS) {
#pragma unroll
                            for (int k = 0; k < 2; ++k) {
                                wv[p][k] = ld_relaxed_u64(qsrc + (size_t)p * (AF_D / 2) + k);
                                all = all && (unsigned)(wv[p][k] >> 32) == (unsigned)(i + 1);
                            }
                        }
                    }
                    return all;
                }, &sh->dead, a.err, 57);
#pragma unroll
                for (int p = 0; p < 4; ++p) {
                    if (p < RS) {
#pragma unroll
                        for (int k = 0; k < 2; ++k) {
                            q4[2 * k] += bf_lo((uint32_t)wv[p][k]);
                            q4[2 * k + 1] += bf_hi((uint32_t)wv[p][k]);
                        }
                    }
                }
            }
            const uint32_t w0 = pack_bf2(q4[0], q4[1]), w1 = pack_bf2(q4[2], q4[3]);
            if (grow < B) *reinterpret_cast<uint2 *>(a.dq_rm + ((size_t)t * B + grow) * AF_D + 4 * lane) = make_uint2(w0, w1);
            const uint32_t doff = (uint32_t)(grow * 256 + (((lane >> 1) ^ (grow & 7)) << 4) + (lane & 1) * 8);
#pragma unroll
            for (int p = 0; p < 4; ++p)
                st_async_f32x2(mapa_u32(my_dqs + doff, (uint32_t)p), __uint_as_float(w0), __uint_as_float(w1), mapa_u32(my_xb1, (uint32_t)p));
            fb_wait_warp(sh->xb + 1, par, &sh->dead, a.err, 55);
            // d h_q[64 rows][8 units] = d q . W_query^T on mma.sync: warp (row tile qm, k quarter kq)
            const int rA = 16 * qm + g4, rB = rA + 8;
            const uint8_t *ra = dqs + rA * 256 + 4 * tig, *rb = dqs + rB * 256 + 4 * tig;
            float cf[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int s2 = 0; s2 < 2; ++s2) {
                const int ch = 2 * (2 * kq + s2);
                const uint32_t a0 = *reinterpret_cast<const uint32_t *>(ra + ((ch ^ (rA & 7)) << 4));
                const uint32_t a1 = *reinterpret_cast<const uint32_t *>(rb + ((ch ^ (rB & 7)) << 4));
                const uint32_t a2 = *reinterpret_cast<const uint32_t *>(ra + (((ch + 1) ^ (rA & 7)) << 4));
                const uint32_t a3 = *reinterpret_cast<const uint32_t *>(rb + (((ch + 1) ^ (rB & 7)) << 4));
                mma_bf16_16816(cf, a0, a1, a2, a3, wqf[s2][0], wqf[s2][1]);
            }
            *reinterpret_cast<float2 *>(dhqp + ((size_t)(kq * PC_ROWS + rA)) * 8 + 2 * tig) = make_float2(cf[0], cf[1]);
            *reinterpret_cast<float2 *>(dhqp + ((size_t)(kq * PC_ROWS + rB)) * 8 + 2 * tig) = make_float2(cf[2], cf[3]);
        }
        __syncthreads();
        if (tid == 0) { pc_stamp(a.dbg, j, i, 4); fb_gstamp(a.dbg, j, i, 4); }
        {
            uint2 dgp = make_uint2(0u, 0u);
            if (uvalid) {
                const float dhq = ((dhqp[(0 * PC_ROWS + ub) * 8 + uk] + dhqp[(1 * PC_ROWS + ub) * 8 + uk]) + dhqp[(2 * PC_ROWS + ub) * 8 + uk]) +
                                  dhqp[(3 * PC_ROWS + ub) * 8 + uk];
                const float dh = dhq + dxd + rec;
                float dcp;
                const float4 d4 = fb_lstm_bwd_point(dh, mult, ga, c_prev, c_new, dc, dcp);
                dc = dcp;
                c_new = c_prev;
                dgp = make_uint2(pack_bf2(d4.x, d4.y), pack_bf2(d4.z, d4.w));
                *reinterpret_cast<uint2 *>(a.gimg + (size_t)par * 4 * FB_QBYTES + gimg_off) = dgp;
                fence_proxy_async_global();
            }
            __syncthreads();
            if (tid == 0) { gbar_arrive(bq_own); pc_stamp(a.dbg, j, i, 5); fb_gstamp(a.dbg, j, i, 5); }
            if (uvalid) *reinterpret_cast<uint2 *>(a.dg_rm + ((size_t)t * B + ub) * 4 * FA_A + 4 * uu) = dgp;
        }
        if (i + 1 == T) break;

        // ============================================================ d x_att_t = d gates_t . W_att[:, ctx | h_att]
        // While warp 0 (TMA) and warp 1 (MMA) stream this CTA's K quarter of the d-gates image, the other 14 warps finish
        // the attention step (conv transpose -> carries -> carry dots) and everything static of step t-1 is requested.
        if (tid < FA_E) {
            dctx[tid] = rvalid ? __ldcs(a.dhc + ((size_t)(t - 1) * B + row) * a.Kp + a.H + tid) + __ldcs(a.dxdall + ((size_t)(t - 1) * B + row) * AE + FA_A + tid) : 0.f;
            ctx32[tid] = rvalid ? __ldcs(a.ctx32 + ((size_t)(t - 1) * B + row) * FA_E + tid) : 0.f;
        }
        if (tid < G.NHP) {
            ws[tid] = tid < n_own ? a.align[((size_t)row * T + (t - 1)) * N + n_lo + tid] : 0.f;
            if (a.d_align) dals[tid] = tid < n_own ? a.d_align[((size_t)row * T + (t - 1)) * N + n_lo + tid] : 0.f;
        }
        // (elect.sync, not `lane == 0`: only then does the compiler treat the single-thread loops as warp-uniform and keep the
        // descriptors in uniform registers - with a divergent branch every UTCHMMA / UBLKCP sits in an ELECT + R2UR.BROADCAST
        // waterfall loop, ~75 cycles per MMA instead of ~10.  16 slabs = two revolutions of the 8-slot ring: slot and phase
        // restart at 0 every step, no state is carried in registers.)
        if (wid == 0) {
            if (elect_one()) {      // TMA producer: this CTA's K quarter of the d-gates image
                // A slab is fetched as soon as ITS two producer CTAs have arrived (per-slab counters, read 16 at a time with relaxed
                // vector loads + one fence): the stream starts under the skew of the 32 producers instead of after the last one.
                // Slabs 0..7 go to their ring slots in any order; slab s >= 8 needs slot s - 8 back from the MMA issuer, which
                // consumes in order (fixed accumulation order: bit-exact run to run).
                const unsigned target = 2u * (unsigned)(i + 1);
                const uint8_t *src = a.gimg + (size_t)par * 4 * FB_QBYTES + (size_t)r * FB_QBYTES;
                uint32_t pending = okw ? 0xffffu : 0u, have = 0u;
                bool first = true;
                const long long t0 = clock64();
                while (pending) {
                    unsigned cnt[16];
#pragma unroll
                    for (int q4 = 0; q4 < 3; ++q4)
                        asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                     : "=r"(cnt[4 * q4]), "=r"(cnt[4 * q4 + 1]), "=r"(cnt[4 * q4 + 2]), "=r"(cnt[4 * q4 + 3])
                                     : "l"(bq_need + 4 * q4)
                                     : "memory");
                    // (the last one is an acquire: everything this thread issues afterwards - the TMA reads - is ordered behind it;
                    // a separate fence.acq_rel.gpu here is a MEMBAR.ALL.GPU on the critical path)
                    asm volatile("ld.acquire.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                                 : "=r"(cnt[12]), "=r"(cnt[13]), "=r"(cnt[14]), "=r"(cnt[15])
                                 : "l"(bq_need + 12)
                                 : "memory");
                    uint32_t ready = 0;
#pragma unroll
                    for (int s = 0; s < 16; ++s)
                        if (cnt[s] >= target) ready |= 1u << s;
                    ready &= pending;
                    if (ready) {
                        fence_proxy_async_global();
                        if (first) {
                            pc_stamp(a.dbg, j, i, 8);
                            fb_gstamp(a.dbg, j, i, 8);
                            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // the ring was used through the generic proxy
                            first = false;
                        }
#pragma unroll 1
                        for (int s = 0; s < 8; ++s) {
                            if (!(ready >> s & 1u)) continue;
                            mbar_expect_tx(sh->full + s, PC_CHUNK_BYTES);
                            tma_bulk_g2s(ring + (size_t)s * PC_CHUNK_BYTES, src + (size_t)s * PC_CHUNK_BYTES, PC_CHUNK_BYTES, sh->full + s);
                        }
                        pending &= ~(ready & 0xffu);
                        have |= ready;
                    }
                    if ((pending & 0xffu) == 0u && (have & 0xff00u) == 0xff00u) break;       // first revolution issued, second one ready
                    if (sh->dead) break;
                    if (clock64() - t0 > FA_WAIT_CYCLES) { sh->dead = 1; atomicCAS(a.err, 0, 58); break; }
                }
                // second revolution of the ring: slab s takes slot s - 8 as soon as the MMA issuer has released it (a shared-memory
                // mbarrier wait - re-polling the global counters here cost an L2 round trip per attempt)
                if (!sh->dead && (have & 0xff00u) == 0xff00u) {
#pragma unroll 1
                    for (int s = 8; s < 16; ++s) {
                        const int slot = s - 8;
                        if (!fa_wait_mbar(sh->empty + slot, 0u, &sh->dead, a.err, 59)) break;
                        mbar_expect_tx(sh->full + slot, PC_CHUNK_BYTES);
                        tma_bulk_g2s(ring + (size_t)slot * PC_CHUNK_BYTES, src + (size_t)s * PC_CHUNK_BYTES, PC_CHUNK_BYTES, sh->full + slot);
                    }
                }
                pc_stamp(a.dbg, j, i, 9);
            }
            __syncwarp();
        } else if (wid == 1) {
            if (elect_one()) {      // MMA issuer
                constexpr uint32_t idesc = umma_idesc_bf16(64, FB_NCOL);
                const uint64_t a0 = umma_desc_sw128(smem_u32(ring)), b0 = umma_desc_sw128(smem_u32(wsm));
                bool ok = okw;
                static_assert(FB_KSLAB == 16, "the issue loop below is unrolled for two revolutions of the 8-slot ring");
                // fully unrolled: slot, phase parity and both descriptors are immediates - the rolled loop spent ~280 cycles per slab
                // on its own bookkeeping (mbarrier wait helper, descriptor arithmetic through R2UR) and bounded the whole stream
#pragma unroll
                for (int s = 0; s < FB_KSLAB; ++s) {
                    const int ring_slot = s & 7;                 // slab s lives in slot s % 8: phase parity 0 for s < 8, 1 for s >= 8
                    if (ok && !mbar_try_wait(sh->full + ring_slot, (uint32_t)(s >> 3))) ok = fa_wait_mbar(sh->full + ring_slot, (uint32_t)(s >> 3), &sh->dead, a.err, 60);
                    if (s == 0) pc_stamp(a.dbg, j, i, 10);
                    if (ok) {
                        tc_fence_after();
                        const uint64_t ad = a0 + (uint64_t)(ring_slot * (PC_CHUNK_BYTES >> 4)), bd = b0 + (uint64_t)(s * (FB_WSLAB_BYTES >> 4));
                        umma_bf16(tmem_base, ad, bd, idesc, s > 0 ? 1u : 0u);
                        umma_bf16(tmem_base, ad + 2, bd + 2, idesc, 1u);
                        umma_bf16(tmem_base, ad + 4, bd + 4, idesc, 1u);
                        umma_bf16(tmem_base, ad + 6, bd + 6, idesc, 1u);
                        umma_commit(sh->empty + ring_slot);
                    }
                }
                if (ok) umma_commit(&sh->tmem_full);
                pc_stamp(a.dbg, j, i, 11);
                // the only thread that waits for the accumulator: everybody else sleeps in the CTA barrier below (warps spinning
                // on mbarriers compete with this thread and the TMA thread for the memory-instruction pipe)
                fa_wait_mbar(&sh->tmem_full, par, &sh->dead, a.err, 61);
            }
            __syncwarp();
        } else {
            const int wt = tid - 64;                                  // 0..447
            if (has_left || has_right) fb_wait_warp(sh->xb + 2, par, &sh->dead, a.err, 56);     // the neighbours' d conv halos are in
            {   // conv transpose: d wcat[c][m] = sum_{f,k} d conv[f][m + 15 - k] wlc[f][c][k]; task = (filter pair, channel, 8 tokens)
                const int ntask = 16 * 2 * G.nblk;
                for (int task = wt; task < ntask; task += 448) {
                    const int fp = task & 15, rest = task >> 4;
                    const int ch = rest / G.nblk, m0 = (rest - ch * G.nblk) * 8;
                    float acc[8];
#pragma unroll
                    for (int q = 0; q < 8; ++q) acc[q] = 0.f;
#pragma unroll
                    for (int ff = 0; ff < 2; ++ff) {
                        const int f = 2 * fp + ff;
                        float x[40];
                        const float4 *xr = reinterpret_cast<const float4 *>(dconvT + f * G.NDS + m0);
#pragma unroll
                        for (int q = 0; q < 10; ++q) {
                            const float4 t4 = xr[q];
                            x[4 * q] = t4.x; x[4 * q + 1] = t4.y; x[4 * q + 2] = t4.z; x[4 * q + 3] = t4.w;
                        }
                        const float *wr = wlc + (f * 2 + ch) * AF_KS;
#pragma unroll
                        for (int k = 0; k < AF_KS; ++k) {
                            const float wk = wr[k];
#pragma unroll
                            for (int q = 0; q < 8; ++q) acc[q] = fmaf(wk, x[q - k + 30], acc[q]);
                        }
                    }
                    float4 *dst = reinterpret_cast<float4 *>(cpart + (fp * 2 + ch) * G.NH + m0);
                    dst[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
                    dst[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
                }
            }
            fb_bar_w14();
            if (wt < 2 * G.NH) {
                const int ch = wt >= G.NH, m = wt - ch * G.NH;
                float s = 0.f;
#pragma unroll
                for (int fp = 0; fp < 16; ++fp) s += cpart[(fp * 2 + ch) * G.NH + m];
                if (ch == 0) dwc[m] = s;
                else dcumc[m] += s;
            }
            fb_bar_w14();
            if (wid == 2) {   // <w_{t-1}, carries> over the own tokens, pushed to every part of the row (this CTA included)
                float p = 0.f;
                for (int n = lane; n < own_len; n += 32) p = fmaf(ws[n], (dwc[n] + dcumc[n]) + dals[n], p);
                p = warp_sum(p);
                if (lane < RS) st_async_f32(mapa_u32(my_xch + 4 * prt, (uint32_t)(gbase + lane)), p, mapa_u32(my_xb0, (uint32_t)(gbase + lane)));
            }
        }
        load_mem(0);            // encoder-memory operand of step t-1's d w phase
        if (uvalid) mult = drop_mult(drop, SITE_ATT, (uint32_t)(t - 1), (uint32_t)(ub + a.row_offset), (uint32_t)uu);
        __syncthreads();
        const bool okt = sh->dead == 0;
        if (tid == 0) { pc_stamp(a.dbg, j, i, 6); fb_gstamp(a.dbg, j, i, 6); }
        if (wid == 0 && elect_one()) {
            if (th_live) {      // tanh tile of step t-1 (lands in ring slots the MMAs have finished reading)
                mbar_expect_tx(&sh->thbar, (uint32_t)n_own * AF_D * 2);
                tma_bulk_g2s(ths, a.th + (((size_t)(t - 1) * B + row) * N + n_lo) * AF_D, (uint32_t)n_own * AF_D * 2, &sh->thbar);
            }
        }
        if (wid >= 4 && okt) {   // TMEM -> the owners' partial tiles.  M = 64: row b in lane (b & 15) of quadrant b >> 4
            const int q = wid & 3, cg3 = (wid >> 2) - 1;
            float vals[16];
            tc_fence_after();
            tmem_ld16(tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(16 * cg3), vals);
            tc_fence_before();
            if (lane < 16) {
                const int b = 16 * q + lane;
#pragma unroll
                for (int n = 0; n < 16; ++n) {
                    const int col = 16 * cg3 + n;                    // compile-time per (cg3 uniform per warp, n unrolled)
                    const int owner = col < 32 ? col >> 3 : (col - 32) >> 2;
                    const int off = (r * 12 + (col < 32 ? col & 7 : 8 + ((col - 32) & 3))) * FB_PLD + b;
                    st_async_f32(mapa_u32(my_pin + 4 * off, (uint32_t)owner), vals[n], mapa_u32(my_xb3, (uint32_t)owner));
                }
            }
        }
        fb_wait_warp(sh->xb + 3, par, &sh->dead, a.err, 62);
        {
            const int o = uk * FB_PLD + ub;
            rec = ((pin[o] + pin[12 * FB_PLD + o]) + pin[24 * FB_PLD + o]) + pin[36 * FB_PLD + o];
            if (tid < 256) {
                const float *cp4 = pin + (8 + ck) * FB_PLD + cb;
                const float cx = ((cp4[0] + cp4[12 * FB_PLD]) + cp4[24 * FB_PLD]) + cp4[36 * FB_PLD];
                if (cb < B)
                    st_relaxed_u64(a.dctxx + ((size_t)(par ^ 1u) * PC_ROWS + cb) * FA_E + 4 * j + ck,
                                   ((unsigned long long)(unsigned)(i + 1) << 32) | (unsigned long long)__float_as_uint(cx));
            }
        }
        if (tid == 0) { pc_stamp(a.dbg, j, i, 7); fb_gstamp(a.dbg, j, i, 7); }
    }
    __syncthreads();
    cluster.sync();          // peers may still be writing into / reading this CTA's shared memory
    if (wid == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(64) : "memory");
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------
// W_att^T slice of CTA j = (cluster c, rank r): [16 slabs][48 rows][128 B] SWIZZLE_128B.  Row n < 32: x_att column of h_att
// unit 32c + n; row n >= 32: ctx column 16c + n - 32.  K = gate row (4 * unit + gate) in [1024 r, 1024 r + 1024).
// Wa_packed: [4A][Ka] fp32, unit-major rows, columns [prenet P | ctx E | h_att A].
__global__ void k_fb_pack_w(const float *__restrict__ Wa_packed, int Ka, int P, __nv_bfloat16 *__restrict__ img) {
    const size_t per_cta = (size_t)FB_KSLAB * FB_NCOL * 64, total = 128 * per_cta;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int j = (int)(i / per_cta);
        const int rem = (int)(i - (size_t)j * per_cta);
        const int slab = rem / (FB_NCOL * 64), rr = rem - slab * FB_NCOL * 64;
        const int n = rr >> 6, cpos = (rr >> 3) & 7, e = rr & 7;
        const int kk = slab * 64 + ((cpos ^ (n & 7)) << 3) + e;
        const int cc = j >> 2, rk = j & 3;
        const int grow = 1024 * rk + kk;
        const int col = n < 32 ? P + FA_E + 32 * cc + n : P + 16 * cc + (n - 32);
        img[i] = __float2bfloat16(Wa_packed[(size_t)grow * Ka + col]);
    }
}
inline size_t fb_wimg_elems() { return (size_t)128 * FB_KSLAB * FB_NCOL * 64; }
inline size_t fb_gimg_bytes() { return (size_t)2 * 4 * FB_QBYTES; }
inline size_t fb_dctxx_words() { return (size_t)2 * PC_ROWS * FA_E; }
inline size_t fb_dqx_words() { return (size_t)2 * PC_ROWS * 4 * (AF_D / 2); }

// CTAs per batch row: 4 when the rows leave half of the grid idle AND a quarter row is still wider than the 15-token conv halo
inline int fb_row_split(int B, int N) { return (B <= 32 && FbGeom(N, 4).NH >= 16) ? 4 : 2; }

// (own shape test: the BPTT chain splits a row over 2 or 4 CTAs, so it reaches N = 320 at B <= 32 where the forward chain,
// two halves per row, stops at 160)
inline bool fb_supported(const Dims &d, int B, int N) {
    static int sms = -1;
    if (sms < 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    if (d.A != FA_A || d.E != FA_E || d.D != AF_D || d.F != AF_F || d.KS != AF_KS) return false;
    if (B < 1 || B > PC_ROWS || N < 1 || sms < 128 || d.P % 8 != 0 || d.H % 8 != 0) return false;
    const int RS = fb_row_split(B, N);
    if (FbGeom(N, RS).NH > ((FA_MAXN / 2 + 7) & ~7)) return false;       // per-CTA token range the kernel's tiles are sized for
    const size_t smem = FbSmem(N, RS).total;
    if (smem > 227 * 1024) return false;
    static size_t cached_smem = 0;
    static bool cached = false;
    if (cached_smem != smem) {
        cached = 4 * max_resident_clusters(k_att_chain_bwd, FB_THREADS, smem, 4, 128) >= 128;
        cached_smem = smem;
    }
    return cached;
}

inline int launch_att_chain_bwd(const FbArgs &a_in, cudaStream_t st) {
    FbArgs a = a_in;
    a.dbg = pc_dbg_buffer() ? pc_dbg_buffer() + 32 * 1024 : nullptr;      // plane 1 (the decoder-LSTM BPTT chain wrote its stamps before)
    const size_t smem = FbSmem(a.N, a.RS).total;
    static size_t configured = 0;
    if (configured < smem) {
        GVX_CUDA(cudaFuncSetAttribute(k_att_chain_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    GVX_CUDA(cudaMemsetAsync(a.bar, 0, 64 * sizeof(unsigned), st));
    GVX_CUDA(cudaMemsetAsync(a.dctxx, 0, fb_dctxx_words() * sizeof(unsigned long long), st));
    GVX_CUDA(cudaMemsetAsync(a.dqx, 0, fb_dqx_words() * sizeof(unsigned long long), st));
    GVX_CUDA(cudaMemsetAsync(a.gimg, 0, fb_gimg_bytes(), st));
    k_att_chain_bwd<<<128, FB_THREADS, smem, st>>>(a);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace gvx
