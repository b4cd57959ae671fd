// genvox_b200 — bf16 mode drivers: packed operand images, teacher-forced forward, BPTT, inference.
// Same entry points as fp32 mode (gvx_api.cu dispatches on gvx_dims.precision); see gvx_bf16.cuh /
// gvx_tc.cuh for the kernels.  Reference lines: Decoder.forward tacotron2.py:365-388, decode :333-363,
// inference :390-414, BPTT = loss.backward() :520.
#pragma once
#include <cublas_v2.h>

#include "gvx_attention_c2.cuh"
#include "gvx_bf16.cuh"
#include "gvx_blas.cuh"
#include "gvx_layout.cuh"
#include "gvx_misc.cuh"
#include "gvx_fused_fwd.cuh"
#include "gvx_fused_bwd.cuh"
#include "gvx_nt_gemm.cuh"
#include "gvx_infer_prenet.cuh"
#include "gvx_persist.cuh"

namespace gvx {

typedef __nv_bfloat16 bf16;

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

struct BfGeom {
    int Kpa, Kpd, Kpq, Kpp, Dp;        // padded K of: att gates, dec gates, query (A), projection (Kp), S4 (D)
    int Ta, Td, Tq, Tp;                // forward row tiles: att, dec gates, query, projection
    int TaT, TdT, TqT;                 // backward row tiles: rows = Ka, Kd, A
    int G4A, G4H;                      // 4A, 4H (already multiples of 128 when A, H % 32 == 0)
    explicit BfGeom(const Dims &d)
        : Kpa(round_up(d.Ka, 64)), Kpd(round_up(d.Kd, 64)), Kpq(round_up(d.A, 64)), Kpp(round_up(d.Kp, 64)), Dp(round_up(d.D, 64)),
          Ta(d.A / 32), Td(d.H / 32), Tq((d.D + 127) / 128), Tp((d.M + 1 + 127) / 128),
          TaT((d.Ka + 127) / 128), TdT((d.Kd + 127) / 128), TqT((d.A + 127) / 128), G4A(round_up(4 * d.A, 64)), G4H(round_up(4 * d.H, 64)) {}
};

inline int check_bf16_dims(const Dims &d, int B) {
    GVX_CHECK(d.M % 8 == 0 && d.E % 8 == 0 && d.A % 32 == 0 && d.H % 32 == 0 && d.P % 8 == 0 && d.D % 8 == 0,
              "bf16 mode: feature dims must be multiples of 8 and the rnn dims multiples of 32");
    GVX_CHECK(B <= 128, "bf16 mode: at most 128 rows per call");
    return 0;
}

inline int tc_pick_ks(int mtiles, int nkb) {
    int ks = 148 / (mtiles > 0 ? mtiles : 1);
    if (ks > 16) ks = 16;
    if (ks > nkb) ks = nkb;
    if (ks < 1) ks = 1;
    return ks;
}

// ---- bf16 part of the packed weights, appended after the fp32 PackedL block (offsets in floats) ----
struct PackedBfL {
    size_t WaI, WdI, WaTI, WdTI, WqI, WqTI, WpgI, WpgRM, WdRM, WdhhI, WdhhTI, WaRecI, WaPRM, WqB, WaRecTI, WdTRM, WaTRM, total;
    PackedBfL(const Dims &d, size_t base) {
        const BfGeom g(d);
        Carver c;
        c.o = base;
        auto img = [&](int tiles, int kpad) { return c.take(((size_t)tiles * TC_M * kpad + 1) / 2); };
        WaI = img(g.Ta, g.Kpa); WdI = img(g.Td, g.Kpd);
        WaTI = img(g.TaT, g.G4A); WdTI = img(g.TdT, g.G4H);
        WqI = img(g.Tq, g.Kpq); WqTI = img(g.TqT, g.Dp);
        WpgI = img(g.Tp, g.Kpp);
        WpgRM = c.take(((size_t)(d.M + 1) * d.Kp + 1) / 2);
        // persistent decoder-LSTM chain (gvx_persist.cuh): unit-major row-major [4H][Kd] copy for the time-batched input
        // GEMMs, resident W_hh slices for the forward chain and W_hh^T slices for BPTT
        WdRM = c.take(((size_t)4 * d.H * d.Kd + 1) / 2);
        WdhhI = c.take((pc_wimg_elems(d.H) + 1) / 2);
        WdhhTI = c.take((pc_wimg_elems(d.H) + 1) / 2);
        // fused attention chain (gvx_fused_fwd.cuh): resident recurrent weights of the attention LSTM, the prenet columns
        // of W_ih as row-major bf16 for the time-batched input GEMM, W_q as row-major bf16
        WaRecI = c.take(fa_wimg_elems() / 2);
        WaPRM = c.take(((size_t)4 * d.A * d.P + 1) / 2);
        WqB = c.take(((size_t)d.D * d.A + 1) / 2);
        // persistent BPTT of the attention chain (gvx_fused_bwd.cuh): resident [ctx | h_att] columns of W_att^T
        WaRecTI = c.take(fb_wimg_elems() / 2);
        // transposed unit-major weights as row-major bf16 ([Kd][4H], [Ka][4A]): B operands of the all-frames d X contractions
        WdTRM = c.take(((size_t)4 * d.H * d.Kd + 1) / 2);
        WaTRM = c.take(((size_t)4 * d.A * d.Ka + 1) / 2);
        total = c.o;
    }
};

int pack_weights_bf16(const Dims &d, const gvx_weights *w, float *packed, cudaStream_t st) {
    const BfGeom g(d);
    const PackedL PL(d);
    const PackedBfL BL(d, PL.total);
    auto pack = [&](int mode, const float *s0, const float *s1, int Mtot, int K, int ld, int HID, int Kih, int tiles, int kpad,
                    size_t off) {
        TcPackW p;
        memset(&p, 0, sizeof(p));
        p.s0 = s0; p.s1 = s1; p.mode = mode; p.Mtot = Mtot; p.K = K; p.ld = ld; p.HID = HID; p.Kih = Kih;
        k_tc_pack_w<<<grid_for((size_t)tiles * TC_M * kpad), 256, 0, st>>>(p, tiles, kpad, (bf16 *)(packed + off));
        GVX_LAUNCHED(1);
    };
    pack(1, w->att_w_ih, w->att_w_hh, 4 * d.A, d.Ka, 0, d.A, d.P + d.E, g.Ta, g.Kpa, BL.WaI);
    pack(1, w->dec_w_ih, w->dec_w_hh, 4 * d.H, d.Kd, 0, d.H, d.A + d.E, g.Td, g.Kpd, BL.WdI);
    pack(2, w->att_w_ih, w->att_w_hh, d.Ka, 4 * d.A, 0, d.A, d.P + d.E, g.TaT, g.G4A, BL.WaTI);
    pack(2, w->dec_w_ih, w->dec_w_hh, d.Kd, 4 * d.H, 0, d.H, d.A + d.E, g.TdT, g.G4H, BL.WdTI);
    pack(0, w->query_w, nullptr, d.D, d.A, d.A, 0, 0, g.Tq, g.Kpq, BL.WqI);
    pack(3, w->query_w, nullptr, d.A, d.D, d.A, 0, 0, g.TqT, g.Dp, BL.WqTI);
    pack(0, packed + PL.Wpg, nullptr, d.M + 1, d.Kp, d.Kp, 0, 0, g.Tp, g.Kpp, BL.WpgI);
    k_to_bf16<<<grid_for((size_t)(d.M + 1) * d.Kp), 256, 0, st>>>(packed + PL.Wpg, d.Kp, (size_t)(d.M + 1), d.Kp,
                                                               (bf16 *)(packed + BL.WpgRM), d.Kp);
    GVX_LAUNCHED(1);
    k_to_bf16<<<grid_for((size_t)4 * d.H * d.Kd), 256, 0, st>>>(packed + PL.Wd, d.Kd, (size_t)4 * d.H, d.Kd, (bf16 *)(packed + BL.WdRM), d.Kd);
    GVX_LAUNCHED(1);
    if (d.H % 64 == 0) {
        k_pc_pack_w<<<grid_for(pc_wimg_elems(d.H)), 256, 0, st>>>(w->dec_w_hh, d.H, d.H, 0, (bf16 *)(packed + BL.WdhhI));
        k_pc_pack_w<<<grid_for(pc_wimg_elems(d.H)), 256, 0, st>>>(w->dec_w_hh, d.H, d.H, 1, (bf16 *)(packed + BL.WdhhTI));
        GVX_LAUNCHED(2);
    }
    k_to_bf16<<<grid_for((size_t)d.D * d.A), 256, 0, st>>>(w->query_w, d.A, (size_t)d.D, d.A, (bf16 *)(packed + BL.WqB), d.A);
    k_to_bf16<<<grid_for((size_t)4 * d.H * d.Kd), 256, 0, st>>>(packed + PL.WdT, 4 * d.H, (size_t)d.Kd, 4 * d.H, (bf16 *)(packed + BL.WdTRM), 4 * d.H);
    k_to_bf16<<<grid_for((size_t)4 * d.A * d.Ka), 256, 0, st>>>(packed + PL.WaT, 4 * d.A, (size_t)d.Ka, 4 * d.A, (bf16 *)(packed + BL.WaTRM), 4 * d.A);
    GVX_LAUNCHED(3);
    if (d.A == FA_A && d.E == FA_E) {
        k_fa_pack_w<<<grid_for(fa_wimg_elems()), 256, 0, st>>>(packed + PL.Wa, d.Ka, d.P, (bf16 *)(packed + BL.WaRecI));
        k_to_bf16<<<grid_for((size_t)4 * d.A * d.P), 256, 0, st>>>(packed + PL.Wa, d.Ka, (size_t)4 * d.A, d.P, (bf16 *)(packed + BL.WaPRM), d.P);
        k_fb_pack_w<<<grid_for(fb_wimg_elems()), 256, 0, st>>>(packed + PL.Wa, d.Ka, d.P, (bf16 *)(packed + BL.WaRecTI));
        GVX_LAUNCHED(3);
    }
    GVX_CUDA(cudaGetLastError());
    return 0;
}

// ---- bf16 training stash -----------------------------------------------------------------------------
struct StashBfL {
    size_t FR, PRE1, PRE2, PM, CA, GA, CD, GD, ALIGN, CUMS, TH, CONVS, OUT, WPREV, CUM, XAI, XDI, XARM, XDRM, HCRM, PA, PD, PQ, ERR,
        SEED, HIMG, BAR, XIMG, MEMB, BAR2, QBUF, HQ, CTX32, total;
    size_t xai_stride, xdi_stride;     // bf16 elements per frame image
    int NPAD, KSa, KSd, KSq;
    StashBfL(const Dims &d, int B, int N, int T) {
        const BfGeom g(d);
        NPAD = tc_npad(B);
        KSa = tc_pick_ks(g.Ta, g.Kpa / TC_KB); KSd = tc_pick_ks(g.Td, g.Kpd / TC_KB); KSq = tc_pick_ks(g.Tq, g.Kpq / TC_KB);
        Carver c;
        const size_t TB = (size_t)T * B, T1B = (size_t)(T + 1) * B;
        FR = c.take(TB * d.M); PRE1 = c.take(TB * d.P); PRE2 = c.take(TB * d.P);
        PM = c.take((size_t)B * N * d.D);
        CA = c.take(T1B * d.A); GA = c.take(TB * 4 * d.A);
        CD = c.take(T1B * d.H); GD = c.take(TB * 4 * d.H);
        ALIGN = c.take((size_t)B * T * N); CUMS = c.take((size_t)B * T * N);
        TH = c.take(TB * N * d.D); CONVS = c.take(TB * N * d.F);
        OUT = c.take(TB * d.OL);
        WPREV = c.take((size_t)B * N); CUM = c.take((size_t)B * N);
        xai_stride = (size_t)g.Kpa * NPAD; xdi_stride = (size_t)g.Kpd * NPAD;
        XAI = c.take((size_t)T * xai_stride / 2); XDI = c.take((size_t)T * xdi_stride / 2);
        XARM = c.take(TB * d.Ka / 2 + 8); XDRM = c.take(TB * d.Kd / 2 + 8); HCRM = c.take(TB * d.Kp / 2 + 8);
        PA = c.take((size_t)KSa * B * g.Ta * TC_M); PD = c.take((size_t)KSd * B * g.Td * TC_M);
        PQ = c.take((size_t)KSq * B * g.Tq * TC_M);
        ERR = c.take(64);
        SEED = c.take(64);
        HIMG = c.take(pc_himg_elems(d.H) / 2);     // [2][H/64][64][64] bf16 ping-pong h_dec image of the persistent chain
        BAR = c.take(64);
        XIMG = c.take(fa_ximg_bytes() / 4);        // ping-pong [h_att | ctx] operand image of the fused attention chain
        MEMB = c.take(((size_t)B * N * d.E + 1) / 2);     // bf16 copy of the encoder memory (context operand)
        BAR2 = c.take(32 * 18);                    // 2 grid barriers + 16 row-group counters, one 128-byte line each
        QBUF = c.take((size_t)2 * 2 * 64 * d.D);   // 64-bit (value, tag) words
        HQ = c.take(2 * fa_hq_words());            // 64-bit (h_att pair, tag) words: the query projection's input exchange
        CTX32 = c.take(TB * d.E);                  // fp32 attention context per frame (softmax backward of the persistent BPTT)
        total = c.o;
    }
};

struct BwdBfL {
    size_t DOUT, DOUTB, DHC, GDI, GAI, DQI, DGDRM, DGARM, DQRM, PDXD, PDXA, PS4, DCD, DCA, DCTX, DE, DCONV, DZ2, DZ1, DPM, DW, DCUM,
        DWA, DWD, DBIAS, PART1, PART2, ONES, TMP, COLP, ERR, GIMG, DXDALL, BAR, GIMGA, DCTXX, DQX, BARA, GWS, total;
    size_t gws_floats;
    size_t pdxd_stride, pdxa_stride;   // floats per ping-pong half
    int NPAD, KSdT, KSaT, KSs4, post_blocks, colchunks;
    BwdBfL(const Dims &d, int B, int N, int T) {
        const BfGeom g(d);
        NPAD = tc_npad(B);
        KSdT = tc_pick_ks(g.TdT, g.G4H / TC_KB); KSaT = tc_pick_ks(g.TaT, g.G4A / TC_KB); KSs4 = tc_pick_ks(g.TqT, g.Dp / TC_KB);
        post_blocks = 148 * 8;
        colchunks = 64;
        Carver c;
        const size_t TB = (size_t)T * B;
        DOUT = c.take(TB * d.OL); DOUTB = c.take(TB * ((d.OL + 7) & ~7) / 2 + 8);     // bf16 copy, row stride rounded up to 8 (TMA)
        DHC = c.take(TB * d.Kp);
        GDI = c.take((size_t)g.G4H * NPAD / 2); GAI = c.take((size_t)g.G4A * NPAD / 2); DQI = c.take((size_t)g.Dp * NPAD / 2);
        DGDRM = c.take(TB * 4 * d.H / 2 + 8); DGARM = c.take(TB * 4 * d.A / 2 + 8); DQRM = c.take(TB * d.D / 2 + 8);
        pdxd_stride = (size_t)KSdT * B * g.TdT * TC_M; pdxa_stride = (size_t)KSaT * B * g.TaT * TC_M;
        PDXD = c.take(2 * pdxd_stride); PDXA = c.take(2 * pdxa_stride);
        PS4 = c.take((size_t)KSs4 * B * g.TqT * TC_M);
        DCD = c.take((size_t)B * d.H); DCA = c.take((size_t)B * d.A);
        DCTX = c.take(TB * d.E);
        DE = c.take(TB * N); DCONV = c.take(TB * N * d.F);
        DZ2 = c.take(TB * d.P); DZ1 = c.take(TB * d.P);
        DPM = c.take((size_t)B * N * d.D);
        DW = c.take((size_t)B * N); DCUM = c.take((size_t)B * N);
        DWA = c.take((size_t)4 * d.A * d.Ka); DWD = c.take((size_t)4 * d.H * d.Kd);
        DBIAS = c.take((size_t)4 * (d.A > d.H ? d.A : d.H));
        PART1 = c.take((size_t)post_blocks * (d.D * d.F + d.D));
        PART2 = c.take((size_t)post_blocks * d.F * 2 * d.KS);
        ONES = c.take(TB);
        TMP = c.take((size_t)(d.M + 1) * d.Kp + 64);
        COLP = c.take((size_t)colchunks * 4 * (d.A > d.H ? d.A : d.H));
        ERR = c.take(64);
        GIMG = c.take(pc_gimg_elems(d.H) / 2);     // [2][4][H/64][64][64] bf16 ping-pong d-gates image of the persistent BPTT chain
        DXDALL = c.take(TB * (d.A + d.E));   // [T][B][A+E] d [h_att | ctx] from the decoder-LSTM input, all frames
        BAR = c.take(64);
        GIMGA = c.take(fb_gimg_bytes() / 4);       // d-gates image of the persistent attention-chain BPTT
        DCTXX = c.take(2 * fb_dctxx_words());      // 64-bit (value, tag) words
        DQX = c.take(2 * fb_dqx_words());
        BARA = c.take(32 * 4);
        gws_floats = (size_t)32 << 20;         // 128 MB: up to 3 partial copies of the largest weight gradient
        GWS = c.take(gws_floats);              // split-K partial tiles of the small weight gradients
        total = c.o;
    }
};

struct InferBfL {
    size_t PM, PRE1, PRE2, CA, CD, Q, WPREV, CUM, OUT, ZERO, FLAGS, XAI, XDI, XPI, PA, PD, PQ, PP, ERR, total;
    size_t xai_stride, xdi_stride;
    int NPAD, KSa, KSd, KSq, KSp;
    InferBfL(const Dims &d, int B, int N, int steps) {
        const BfGeom g(d);
        NPAD = tc_npad(B);
        KSa = tc_pick_ks(g.Ta, g.Kpa / TC_KB); KSd = tc_pick_ks(g.Td, g.Kpd / TC_KB); KSq = tc_pick_ks(g.Tq, g.Kpq / TC_KB);
        KSp = tc_pick_ks(g.Tp, g.Kpp / TC_KB);
        Carver c;
        PM = c.take((size_t)B * N * d.D);
        PRE1 = c.take((size_t)B * d.P); PRE2 = c.take((size_t)B * d.P);
        CA = c.take((size_t)B * d.A); CD = c.take((size_t)B * d.H);
        Q = c.take((size_t)B * d.D);
        WPREV = c.take((size_t)B * N); CUM = c.take((size_t)B * N);
        OUT = c.take((size_t)steps * B * d.OL);
        ZERO = c.take((size_t)B * d.OL);
        FLAGS = c.take(64);
        xai_stride = (size_t)g.Kpa * NPAD; xdi_stride = (size_t)g.Kpd * NPAD;
        XAI = c.take(2 * xai_stride / 2); XDI = c.take(2 * xdi_stride / 2);
        XPI = c.take((size_t)g.Kpp * NPAD / 2);
        PA = c.take((size_t)KSa * B * g.Ta * TC_M); PD = c.take((size_t)KSd * B * g.Td * TC_M);
        PQ = c.take((size_t)KSq * B * g.Tq * TC_M); PP = c.take((size_t)KSp * B * g.Tp * TC_M);
        ERR = c.take(64);
        total = c.o;
    }
};

// one tcgen05 gate GEMM: P[KS][B][tiles*128] = Wimg . Ximg
inline int run_tc(const bf16 *Wimg, const bf16 *Ximg, float *P, int tiles, int kpad, int KS, int B, int *err, cudaStream_t st) {
    TcGemmArgs a;
    memset(&a, 0, sizeof(a));
    a.Wimg = Wimg; a.Ximg = Ximg; a.P = P; a.Kpad = kpad; a.B = B; a.ldp = tiles * TC_M; a.KS = KS; a.err = err;
    return launch_tc_gemm(a, tiles, st);
}

inline int run_bf_lstm_fwd(const Dims &d, const float *packed, int which, const float *P, int KS, int tiles, const float *c_prev,
                           float *c_out, float *gates_out, const BfDsts &h_dst, int B, uint64_t seed, int t, int training,
                           int row_offset, cudaStream_t st) {
    const PackedL PL(d);
    BfLstmFwd a;
    memset(&a, 0, sizeof(a));
    a.P = P; a.KS = KS; a.ldp = tiles * TC_M;
    a.bias = packed + (which == 0 ? PL.ba : PL.bd);
    a.c_prev = c_prev; a.c_out = c_out; a.gates_out = gates_out; a.h_dst = h_dst;
    a.drop = make_drop(seed, which == 0 ? d.p_att : d.p_dec, training);
    a.site = which == 0 ? SITE_ATT : SITE_DEC;
    a.t = (uint32_t)t; a.row_offset = row_offset; a.B = B; a.HID = which == 0 ? d.A : d.H;
    GVX_CUDA(launch_pdl(k_bf_lstm_fwd, dim3(grid_for((size_t)B * a.HID)), dim3(256), 0, st, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

// gate GEMM + LSTM cell: fused cluster kernel when the K range splits in 4 (GVX_FUSED_LSTM=0: GEMM -> partials -> cell kernel)
inline int run_lstm_bf16(const Dims &d, const float *packed, int which, const bf16 *Wimg, const bf16 *Ximg, float *P, int KS,
                         int tiles, int kpad, const float *c_prev, float *c_out, float *gates_out, const BfDsts &h_dst, int B,
                         uint64_t seed, int t, int training, int row_offset, int *err, cudaStream_t st) {
    if (tc_fused_lstm_enabled() && kpad / TC_KB >= 4 && 4 * tiles <= 148) {
        const PackedL PL(d);
        TcLstmArgs p;
        memset(&p, 0, sizeof(p));
        p.g.Wimg = Wimg; p.g.Ximg = Ximg; p.g.P = nullptr; p.g.Kpad = kpad; p.g.B = B; p.g.ldp = tiles * TC_M; p.g.KS = 4; p.g.err = err;
        p.bias = packed + (which == 0 ? PL.ba : PL.bd);
        p.c_prev = c_prev; p.c_out = c_out; p.gates_out = gates_out; p.h_dst = h_dst;
        p.drop = make_drop(seed, which == 0 ? d.p_att : d.p_dec, training);
        p.site = which == 0 ? SITE_ATT : SITE_DEC;
        p.t = (uint32_t)t; p.row_offset = row_offset; p.HID = which == 0 ? d.A : d.H;
        return launch_tc_gemm_lstm(p, tiles, st);
    }
    GVX_TRY(run_tc(Wimg, Ximg, P, tiles, kpad, KS, B, err, st));
    return run_bf_lstm_fwd(d, packed, which, P, KS, tiles, c_prev, c_out, gates_out, h_dst, B, seed, t, training, row_offset, st);
}

inline int check_tc_err(int *err_dev, cudaStream_t st, const char *what) {
    int h = 0;
    GVX_CUDA(cudaMemcpyAsync(&h, err_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    GVX_CUDA(cudaStreamSynchronize(st));
    if (h) {
        snprintf(g_err, sizeof(g_err), "%s: tcgen05 pipeline timeout (code %d)", what, h);
        return 1;
    }
    return 0;
}

// bf16 x bf16 -> fp32 time-batched GEMMs (plain library GEMMs): row-major C[M,N] = op(A) . op(B)
inline int gemm_tn_bf16(cudaStream_t st, int M, int N, int K, const bf16 *A, int lda, const bf16 *Bm, int ldb, float *Cm, int ldc) {
    cublasHandle_t h;
    GVX_TRY(blas(&h, st));
    const float alpha = 1.f, beta = 0.f;
    cublasStatus_t s = cublasGemmEx(h, CUBLAS_OP_N, CUBLAS_OP_T, N, M, K, &alpha, Bm, CUDA_R_16BF, ldb, A, CUDA_R_16BF, lda, &beta, Cm,
                                    CUDA_R_32F, ldc, CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    if (s != CUBLAS_STATUS_SUCCESS) { snprintf(g_err, sizeof(g_err), "cublasGemmEx(TN bf16) failed: %d", (int)s); return 1; }
    return 0;
}
// C[M,N] = A[M,K] . W[N,K]^T
inline int gemm_nt_bf16(cudaStream_t st, int M, int N, int K, const bf16 *A, int lda, const bf16 *Wm, int ldw, float *Cm, int ldc) {
    cublasHandle_t h;
    GVX_TRY(blas(&h, st));
    const float alpha = 1.f, beta = 0.f;
    cublasStatus_t s = cublasGemmEx(h, CUBLAS_OP_T, CUBLAS_OP_N, N, M, K, &alpha, Wm, CUDA_R_16BF, ldw, A, CUDA_R_16BF, lda, &beta, Cm,
                                    CUDA_R_32F, ldc, CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    if (s != CUBLAS_STATUS_SUCCESS) { snprintf(g_err, sizeof(g_err), "cublasGemmEx(NT bf16) failed: %d", (int)s); return 1; }
    return 0;
}

// C[M,N] = A[M,K] . Wm[K,N]   (all row-major)
inline int gemm_nn_bf16(cudaStream_t st, int M, int N, int K, const bf16 *A, int lda, const bf16 *Wm, int ldw, float *Cm, int ldc) {
    cublasHandle_t h;
    GVX_TRY(blas(&h, st));
    const float alpha = 1.f, beta = 0.f;
    cublasStatus_t s = cublasGemmEx(h, CUBLAS_OP_N, CUBLAS_OP_N, N, M, K, &alpha, Wm, CUDA_R_16BF, ldw, A, CUDA_R_16BF, lda, &beta, Cm,
                                    CUDA_R_32F, ldc, CUBLAS_COMPUTE_32F, CUBLAS_GEMM_DEFAULT);
    if (s != CUBLAS_STATUS_SUCCESS) { snprintf(g_err, sizeof(g_err), "cublasGemmEx(NN bf16) failed: %d", (int)s); return 1; }
    return 0;
}

// The all-frames contractions run on the own tcgen05 GEMM (gvx_nt_gemm.cuh).  GVX_OWN_GEMM=0 sends them to cuBLAS instead
// (comparison runs only).
inline bool own_gemm() {
    static int on = -1;
    if (on < 0) {
        const char *e = getenv("GVX_OWN_GEMM");
        on = (e && e[0] == '0') ? 0 : 1;
    }
    return on == 1;
}
// C[M,N] = A[M,K] . W[N,K]^T
inline int gemm_nt(cudaStream_t st, int M, int N, int K, const bf16 *A, int lda, const bf16 *Wm, int ldw, float *Cm, int ldc, int *err) {
    if (own_gemm() && K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0) return nt_gemm_bf16(st, M, N, K, A, lda, Wm, ldw, Cm, ldc, err);
    return gemm_nt_bf16(st, M, N, K, A, lda, Wm, ldw, Cm, ldc);
}

__global__ void k_add_bias_rows(float *x, size_t rows, int cols, int ld, const float *__restrict__ bias) {
    const size_t total = rows * cols;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / cols;
        const int c = (int)(i - r * cols);
        x[r * ld + c] += bias[c];
    }
}

// the fused persistent attention chains (forward + BPTT) go together: they share the bf16 / swizzled tanh stash
inline bool fused_chains_ok(const Dims &d, int B, int N) {
    return pc_enabled() && pc_supported(d.H, B) && fa_enabled() && fa_supported(d, B, N) && fb_supported(d, B, N);
}
// the persistent BPTT attention chain behind a PER-STEP forward chain (shapes the persistent forward does not cover, e.g.
// configs[4]: B = 32, N = 300): the per-step attention kernel then writes the stashes in the formats the BPTT chain reads
// (bf16 / swizzled tanh rows, fp32 context per frame) and the bf16 copy of the encoder memory is made up front
inline bool fused_bwd_only_ok(const Dims &d, int B, int N) {
    return pc_enabled() && pc_supported(d.H, B) && fa_enabled() && !fa_supported(d, B, N) && fb_supported(d, B, N) &&
           attention_fwd_uses_c2(AttnShape{B, N, d.D, d.E, d.F, d.KS});
}

// ======================================================================================= forward (training)
int train_fwd_bf16(const Dims &d, const gvx_weights *w, const float *packed, const float *memory, const float *mel_in,
                          const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training, int row_offset,
                          float *mel_out, float *gate_out, float *align_out, float *s, cudaStream_t st) {
    GVX_TRY(check_bf16_dims(d, B));
    const BfGeom g(d);
    const PackedL PL(d);
    const PackedBfL BL(d, PL.total);
    const StashBfL S(d, B, N, T);
    const int NPAD = S.NPAD;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H;
    bf16 *XAI = (bf16 *)(s + S.XAI), *XDI = (bf16 *)(s + S.XDI), *XARM = (bf16 *)(s + S.XARM), *XDRM = (bf16 *)(s + S.XDRM),
         *HCRM = (bf16 *)(s + S.HCRM);
    int *err = (int *)(s + S.ERR);
    const bf16 *WaI = (const bf16 *)(packed + BL.WaI), *WdI = (const bf16 *)(packed + BL.WdI), *WqI = (const bf16 *)(packed + BL.WqI);
    // persistent decoder-LSTM chain: its input part does not depend on the decoder LSTM under teacher forcing, so the
    // attention chain runs first for all frames and the decoder-LSTM recurrence follows in ONE launch (gvx_persist.cuh)
    const bool pc = pc_enabled() && pc_supported(d.H, B);
    // fused attention chain: attention LSTM + query + attention of all frames in ONE persistent launch (gvx_fused_fwd.cuh)
    const bool fa = fused_chains_ok(d, B, N);
    const bool fbo = !fa && fused_bwd_only_ok(d, B, N);      // per-step forward, persistent BPTT attention chain

    ProfScope *ps_setup = new ProfScope(PS_SETUP, st);
    GVX_CUDA(cudaMemsetAsync(err, 0, 64 * sizeof(float), st));
    // operand images start as zeros: K padding, ctx_{-1} = h_{-1} = 0 (tacotron2.py:303-315)
    if (!fa) {
        GVX_CUDA(cudaMemsetAsync(XAI, 0, (size_t)T * S.xai_stride * sizeof(bf16), st));
        GVX_CUDA(cudaMemsetAsync(XDI, 0, (size_t)T * S.xdi_stride * sizeof(bf16), st));
    } else {
        GVX_CUDA(cudaMemsetAsync(s + S.XIMG, 0, fa_ximg_bytes(), st));
    }
    if (fa || fbo) {
        k_to_bf16<<<grid_for((size_t)B * N * d.E), 256, 0, st>>>(memory, d.E, (size_t)B * N, d.E, (bf16 *)(s + S.MEMB), d.E);
        GVX_LAUNCHED(1);
    }
    GVX_CUDA(cudaMemsetAsync(XARM, 0, (size_t)B * d.Ka * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(XDRM, 0, (size_t)B * d.Kd * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CA, 0, BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.WPREV, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CUM, 0, (size_t)B * N * sizeof(float), st));
    k_pack_frames<<<grid_for((size_t)T * B * d.M), 256, 0, st>>>(mel_in, B, d.M, T, s + S.FR);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    {
        BfDsts bf;
        memset(&bf, 0, sizeof(bf));
        if (!fa) bf.d[bf.n++] = BfDst{XAI, 1, 0, NPAD, (long long)S.xai_stride};
        bf.d[bf.n++] = BfDst{XARM, 2, 0, d.Ka, (long long)B * d.Ka};
        GVX_TRY(run_prenet(d, w, s + S.FR, d.M, T * B, B, seed, 0, row_offset, s + S.PRE1, s + S.PRE2, st, &bf));
    }
    GVX_TRY(run_processed_memory(d, w, memory, B, N, s + S.PM, st));
    delete ps_setup;

    if (fa) {
        {   // prenet part of the attention-LSTM gate pre-activations for all frames (tacotron2.py:338-340)
            ProfScope ps(PS_ATT_LSTM, st);
            GVX_TRY(gemm_nt(st, T * B, 4 * d.A, d.P, XARM, d.Ka, (const bf16 *)(packed + BL.WaPRM), d.P, s + S.GA, 4 * d.A, err));
        }
        ProfScope ps(PS_ATTENTION, st);
        FaArgs f;
        memset(&f, 0, sizeof(f));
        f.Wimg = (const bf16 *)(packed + BL.WaRecI);
        f.pre = s + S.GA; f.bias = packed + PL.ba;
        f.ximg = (uint8_t *)(s + S.XIMG);
        f.c_stash = s + S.CA; f.gates_stash = s + S.GA;
        f.xdrm = XDRM; f.xarm = XARM; f.hcrm = HCRM;
        f.Kd = d.Kd; f.Ka = d.Ka; f.Kp = d.Kp; f.P = d.P; f.H = d.H;
        f.Wq = (const bf16 *)(packed + BL.WqB);
        f.pm = s + S.PM; f.memb = (const bf16 *)(s + S.MEMB);
        f.wlc = w->loc_conv_w; f.wldT = packed + PL.wldT; f.v = w->v_w; f.lengths = mem_lengths;
        f.align_out = s + S.ALIGN; f.cum_stash = s + S.CUMS; f.th_stash = s + S.TH; f.th_bf16 = 1; f.conv_stash = s + S.CONVS; f.ctx32_stash = s + S.CTX32;
        f.bar = (unsigned *)(s + S.BAR2); f.qbuf = (unsigned long long *)(s + S.QBUF); f.hq = (unsigned long long *)(s + S.HQ); f.err = err;
        f.drop = make_drop(seed, d.p_att, training);
        f.row_offset = row_offset; f.B = B; f.N = N; f.T = T;
        GVX_TRY(launch_att_chain_fwd(f, st));
    }
    pdl_barrier_next();
    for (int t = 0; t < T && !fa; ++t) {
        const bool more = t + 1 < T;
        bf16 *xa = XAI + (size_t)t * S.xai_stride, *xd = XDI + (size_t)t * S.xdi_stride;
        bf16 *xa_n = more ? XAI + (size_t)(t + 1) * S.xai_stride : nullptr, *xd_n = more ? XDI + (size_t)(t + 1) * S.xdi_stride : nullptr;
        bf16 *xarm_n = more ? XARM + (size_t)(t + 1) * B * d.Ka : nullptr, *xdrm = XDRM + (size_t)t * B * d.Kd;
        bf16 *xdrm_n = more ? XDRM + (size_t)(t + 1) * B * d.Kd : nullptr, *hcrm = HCRM + (size_t)t * B * d.Kp;
        {   // attention LSTM (tacotron2.py:338-341)
            ProfScope ps(PS_ATT_LSTM, st);
            BfDsts h;
            memset(&h, 0, sizeof(h));
            add_img(h, xd, 0, NPAD); add_rm(h, xdrm, 0, d.Kd);
            add_img(h, xa_n, d.P + d.E, NPAD); add_rm(h, xarm_n, d.P + d.E, d.Ka);
            GVX_TRY(run_lstm_bf16(d, packed, 0, WaI, xa, s + S.PA, S.KSa, g.Ta, g.Kpa, s + S.CA + t * BA, s + S.CA + (t + 1) * BA,
                                  s + S.GA + (size_t)t * 4 * BA, h, B, seed, t, training, row_offset, err, st));
        }
        {   // query projection (:98): X = the h_att prefix of the decoder-LSTM operand image
            ProfScope ps(PS_QUERY, st);
            GVX_TRY(run_tc(WqI, xd, s + S.PQ, g.Tq, g.Kpq, S.KSq, B, err, st));
        }
        {   // attention (:344-353)
            ProfScope ps(PS_ATTENTION, st);
            AttnFwdArgs a;
            memset(&a, 0, sizeof(a));
            a.s = AttnShape{B, N, d.D, d.E, d.F, d.KS};
            a.q = src_split(s + S.PQ, g.Tq * TC_M, S.KSq, (long long)B * g.Tq * TC_M);
            a.pm = s + S.PM; a.memory = memory;
            a.wlc = w->loc_conv_w; a.wldT = packed + PL.wldT; a.v = w->v_w; a.lengths = mem_lengths;
            a.w_prev = s + S.WPREV; a.cum = s + S.CUM;
            a.align_out = s + S.ALIGN + (size_t)t * N; a.align_bstride = (long long)T * N;
            a.cum_stash = s + S.CUMS + (size_t)t * N;
            a.ctx_out = nullptr; a.ctx_ld = d.E;
            if (!pc) add_img(a.ctx_bf, xd, d.A, NPAD);
            add_rm(a.ctx_bf, xdrm, d.A, d.Kd);
            add_img(a.ctx_bf, xa_n, d.P, NPAD); add_rm(a.ctx_bf, xarm_n, d.P, d.Ka);
            add_rm(a.ctx_bf, hcrm, d.H, d.Kp);
            a.th_stash = s + S.TH + (size_t)t * B * N * d.D;
            if (fbo) {
                a.th_bf16 = 1;
                a.th_stash = reinterpret_cast<float *>(reinterpret_cast<bf16 *>(s + S.TH) + (size_t)t * B * N * d.D);
                a.ctx_out = s + S.CTX32 + (size_t)t * B * d.E;
            }
            a.conv_stash = s + S.CONVS + (size_t)t * B * N * d.F;
            GVX_TRY(launch_attention_fwd_best(a, st));
        }
        if (!pc) {   // decoder LSTM (:355-358)
            ProfScope ps(PS_DEC_LSTM, st);
            BfDsts h;
            memset(&h, 0, sizeof(h));
            add_rm(h, hcrm, 0, d.Kp);
            add_img(h, xd_n, d.A + d.E, NPAD); add_rm(h, xdrm_n, d.A + d.E, d.Kd);
            GVX_TRY(run_lstm_bf16(d, packed, 1, WdI, xd, s + S.PD, S.KSd, g.Td, g.Kpd, s + S.CD + t * BH, s + S.CD + (t + 1) * BH,
                                  s + S.GD + (size_t)t * 4 * BH, h, B, seed, t, training, row_offset, err, st));
        }
    }
    if (pc) {   // decoder LSTM (:355-358) for all frames: time-batched input part, then the persistent recurrence
        {
            ProfScope ps(PS_DEC_IN_GEMM, st);
            GVX_TRY(gemm_nt(st, T * B, 4 * d.H, d.A + d.E, XDRM, d.Kd, (const bf16 *)(packed + BL.WdRM), d.Kd, s + S.GD, 4 * d.H, err));
        }
        ProfScope ps(PS_DEC_LSTM, st);
        GVX_CUDA(cudaMemsetAsync(s + S.HIMG, 0, pc_himg_elems(d.H) * sizeof(bf16), st));
        PcFwdArgs f;
        memset(&f, 0, sizeof(f));
        f.Wimg = (const bf16 *)(packed + BL.WdhhI);
        f.pre = s + S.GD; f.bias = packed + PL.bd;
        f.himg = (bf16 *)(s + S.HIMG);
        f.c_stash = s + S.CD; f.gates_stash = s + S.GD;
        f.out[0] = PcOut{HCRM, d.Kp, 0, 0, (long long)B * d.Kp};
        f.out[1] = PcOut{XDRM, d.Kd, d.A + d.E, 1, (long long)B * d.Kd};
        f.bar = (unsigned *)(s + S.BAR); f.err = err;
        f.drop = make_drop(seed, d.p_dec, training);
        f.site = SITE_DEC; f.row_offset = row_offset; f.B = B; f.T = T; f.H = d.H;
        GVX_TRY(launch_lstm_chain_fwd(f, st));
    }
    ProfScope ps_out(PS_OUTPUT, st);
    // mel / gate projections for all frames (:360-362): [T*B, H+E] bf16 . Wpg^T
    GVX_TRY(gemm_nt(st, T * B, d.M + 1, d.Kp, HCRM, d.Kp, (const bf16 *)(packed + BL.WpgRM), d.Kp, s + S.OUT, d.OL, err));
    k_add_bias_rows<<<grid_for((size_t)T * B * (d.M + 1)), 256, 0, st>>>(s + S.OUT, (size_t)T * B, d.M + 1, d.OL, packed + PL.bpg);
    GVX_LAUNCHED(1);
    k_unpack_out<<<grid_for((size_t)B * (d.M + 1) * T), 256, 0, st>>>(s + S.OUT, B, d.M, d.OL, T, T, mel_out, gate_out);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_CUDA(cudaMemcpyAsync(align_out, s + S.ALIGN, (size_t)B * T * N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_TRY(latch_record(err, 1, 1, st));
    GVX_LAUNCHED(1);
    return 0;
}

inline int run_bf_lstm_bwd(const Dims &d, int which, const SrcSum &s0, const SrcSum &s1, const SrcSum &s2, const float *gates,
                           const float *c_prev, const float *c_new, float *dc, const BfDsts &dg, int B, uint64_t seed, int t,
                           int training, int row_offset, const SrcSum *dpre_src, const float *pre2, float *dz2, cudaStream_t st) {
    BfLstmBwd a;
    memset(&a, 0, sizeof(a));
    a.s0 = s0; a.s1 = s1; a.s2 = s2;
    a.drop = make_drop(seed, which == 0 ? d.p_att : d.p_dec, training);
    a.site = which == 0 ? SITE_ATT : SITE_DEC;
    a.t = (uint32_t)t; a.row_offset = row_offset; a.B = B; a.HID = which == 0 ? d.A : d.H;
    a.gates = gates; a.c_prev = c_prev; a.c_new = c_new; a.dc = dc; a.dg_dst = dg;
    a.main_blocks = grid_for((size_t)B * a.HID);
    int extra = 0;
    if (dpre_src) {
        a.dpre_src = *dpre_src; a.pre2 = pre2; a.dz2 = dz2; a.P = d.P;
        extra = grid_for((size_t)B * d.P);
    }
    GVX_CUDA(launch_pdl(k_bf_lstm_bwd, dim3(a.main_blocks + extra), dim3(256), 0, st, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

// attention-LSTM cell backward of one step with d q . W_query computed inside (k_bf_lstm_bwd_q)
inline int run_bf_lstm_bwd_q(const Dims &d, const bf16 *dq_rm, const float *WqT, const SrcSum &s1, const SrcSum &s2, const float *gates,
                             const float *c_prev, const float *c_new, float *dc, const BfDsts &dg, int B, uint64_t seed, int t,
                             int training, int row_offset, const SrcSum *dpre_src, const float *pre2, float *dz2, cudaStream_t st) {
    BfLstmBwdQ q;
    memset(&q, 0, sizeof(q));
    BfLstmBwd &a = q.p;
    a.s1 = s1; a.s2 = s2;
    a.drop = make_drop(seed, d.p_att, training);
    a.site = SITE_ATT;
    a.t = (uint32_t)t; a.row_offset = row_offset; a.B = B; a.HID = d.A;
    a.gates = gates; a.c_prev = c_prev; a.c_new = c_new; a.dc = dc; a.dg_dst = dg;
    a.main_blocks = (d.A + LBQ_UB - 1) / LBQ_UB;
    int extra = 0;
    if (dpre_src) {
        a.dpre_src = *dpre_src; a.pre2 = pre2; a.dz2 = dz2; a.P = d.P;
        extra = grid_for((size_t)B * d.P);
        if (extra > 64) extra = 64;
    }
    q.dq_rm = dq_rm; q.WqT = WqT; q.D = d.D;
    const size_t smem = ((size_t)((LBQ_UB * (d.D + 1) + 3) & ~3) + (size_t)d.D * (((B + 1) & ~1) + 2)) * sizeof(float);
    static size_t configured = 0;
    if (smem > configured) {
        GVX_CUDA(cudaFuncSetAttribute(k_bf_lstm_bwd_q, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    GVX_CUDA(launch_pdl(k_bf_lstm_bwd_q, dim3(a.main_blocks + extra), dim3(LBQ_THREADS), smem, st, q));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

// ======================================================================================= backward (BPTT)
int train_bwd_bf16(const Dims &d, const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths,
                   int B, int N, int T, uint64_t seed, int training, int row_offset, const float *d_mel, const float *d_gate,
                   const float *d_align, const float *s, float *x, const gvx_grads *g, float *d_memory, cudaStream_t st) {
    GVX_TRY(check_bf16_dims(d, B));
    const BfGeom gm(d);
    const PackedL PL(d);
    const PackedBfL BL(d, PL.total);
    const StashBfL S(d, B, N, T);
    const BwdBfL W(d, B, N, T);
    const int NPAD = W.NPAD, TB = T * B;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H, BE = (size_t)B * d.E;
    const bf16 *WaTI = (const bf16 *)(packed + BL.WaTI), *WdTI = (const bf16 *)(packed + BL.WdTI), *WqTI = (const bf16 *)(packed + BL.WqTI);
    const bf16 *XARM = (const bf16 *)(s + S.XARM), *XDRM = (const bf16 *)(s + S.XDRM), *HCRM = (const bf16 *)(s + S.HCRM);
    bf16 *GDI = (bf16 *)(x + W.GDI), *GAI = (bf16 *)(x + W.GAI), *DQI = (bf16 *)(x + W.DQI);
    bf16 *DGDRM = (bf16 *)(x + W.DGDRM), *DGARM = (bf16 *)(x + W.DGARM), *DQRM = (bf16 *)(x + W.DQRM), *DOUTB = (bf16 *)(x + W.DOUTB);
    int *err = (int *)(x + W.ERR);
    const int ldd = gm.TdT * TC_M, lda = gm.TaT * TC_M, lds4 = gm.TqT * TC_M;

    GVX_CUDA(cudaMemsetAsync(err, 0, 64 * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DW, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCUM, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(x + W.DCA, 0, BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(GDI, 0, (size_t)gm.G4H * NPAD * sizeof(bf16), st));     // K / row padding of the operand images
    GVX_CUDA(cudaMemsetAsync(GAI, 0, (size_t)gm.G4A * NPAD * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(DQI, 0, (size_t)gm.Dp * NPAD * sizeof(bf16), st));
    k_fill_f32<<<grid_for((size_t)TB), 256, 0, st>>>(x + W.ONES, (size_t)TB, 1.f);
    GVX_LAUNCHED(1);
    k_pack_dout<<<grid_for((size_t)TB * d.OL), 256, 0, st>>>(d_mel, d_gate, B, d.M, d.OL, T, x + W.DOUT);
    GVX_LAUNCHED(1);
    const int OLB = (d.OL + 7) & ~7;          // row stride of the bf16 copy: a multiple of 8 elements (16-byte rows for TMA)
    k_to_bf16<<<grid_for((size_t)TB * d.OL), 256, 0, st>>>(x + W.DOUT, d.OL, (size_t)TB, d.OL, DOUTB, OLB);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_TRY(gemm_nn(st, TB, d.Kp, d.M + 1, x + W.DOUT, d.OL, packed + PL.Wpg, d.Kp, x + W.DHC, d.Kp, 0.f));

    const bool pc = pc_enabled() && pc_supported(d.H, B);
    const int AE = d.A + d.E;
    if (pc) {
        {   // BPTT of the decoder-LSTM recurrence for all frames in one persistent launch (gvx_persist.cuh)
            ProfScope ps(PS_BWD_DEC_POINT, st);
            GVX_CUDA(cudaMemsetAsync(x + W.GIMG, 0, pc_gimg_elems(d.H) * sizeof(bf16), st));
            PcBwdArgs a;
            memset(&a, 0, sizeof(a));
            a.Wimg = (const bf16 *)(packed + BL.WdhhTI);
            a.gimg = (bf16 *)(x + W.GIMG);
            a.dh_ext = x + W.DHC; a.dh_ld = d.Kp; a.dh_tstride = (long long)B * d.Kp;
            a.gates_stash = s + S.GD; a.c_stash = s + S.CD; a.dg_rm = DGDRM;
            a.bar = (unsigned *)(x + W.BAR); a.err = err;
            a.drop = make_drop(seed, d.p_dec, training);
            a.site = SITE_DEC; a.row_offset = row_offset; a.B = B; a.T = T; a.H = d.H;
            GVX_TRY(launch_lstm_chain_bwd(a, st));
        }
        {   // d [h_att_t | ctx_t] from the decoder-LSTM input, all frames: d gates_dec . W_ih
            ProfScope ps(PS_BWD_DEC_GEMM, st);
            if (own_gemm()) GVX_TRY(nt_gemm_bf16(st, TB, AE, 4 * d.H, DGDRM, 4 * d.H, (const bf16 *)(packed + BL.WdTRM), 4 * d.H, x + W.DXDALL, AE, err));
            else GVX_TRY(gemm_nn_bf16(st, TB, AE, 4 * d.H, DGDRM, 4 * d.H, (const bf16 *)(packed + BL.WdRM), d.Kd, x + W.DXDALL, AE));
        }
    }

    // OPT-IN (GVX_S4_FUSED=1): measured on B200 at configs[2] the folded kernel is SLOWER than GEMM + pointwise (phase 13.3 ms
    // vs 10.6 ms per train step, whole step 73.1 vs 65.8 ms): its 128 blocks serialise staging, contraction and the
    // latency-bound cell backward, while the two-launch version overlaps them through programmatic dependent launch
    static const bool s4_fused = getenv("GVX_S4_FUSED") && getenv("GVX_S4_FUSED")[0] == '1';
    // d q . W_query folded into the 2-CTA cluster attention-backward kernel (its conv-transpose phase leaves 320 threads idle):
    // one launch less per step.  GVX_DHQ_FOLDED=0 restores the separate engine GEMM.
    static const bool dhq_env = !(getenv("GVX_DHQ_FOLDED") && getenv("GVX_DHQ_FOLDED")[0] == '0');
    const bool dhq_folded = dhq_env && !s4_fused && d.A % 16 == 0 && d.A <= 1024 && attention_bwd_uses_c2(AttnShape{B, N, d.D, d.E, d.F, d.KS});
    // the fused forward chain left a bf16 copy of the encoder memory in the stash: operand of d w in the attention backward
    const bool fb = fused_chains_ok(d, B, N) || fused_bwd_only_ok(d, B, N);
    const bool have_memb = fb;
    if (fb) {   // BPTT of the attention chain for all frames in one persistent launch (gvx_fused_bwd.cuh)
        ProfScope ps(PS_BWD_ATTENTION, st);
        FbArgs f;
        memset(&f, 0, sizeof(f));
        f.Wimg = (const bf16 *)(packed + BL.WaRecTI);
        f.gimg = (uint8_t *)(x + W.GIMGA);
        f.WqB = (const bf16 *)(packed + BL.WqB);
        f.gates_stash = s + S.GA; f.c_stash = s + S.CA;
        f.dxdall = x + W.DXDALL; f.dhc = x + W.DHC; f.Kp = d.Kp; f.H = d.H;
        f.d_align = d_align; f.align = s + S.ALIGN; f.ctx32 = s + S.CTX32;
        f.th = (const bf16 *)(s + S.TH); f.memb = (const bf16 *)(s + S.MEMB);
        f.wlc = w->loc_conv_w; f.wldT = packed + PL.wldT; f.v = w->v_w; f.lengths = mem_lengths;
        f.dg_rm = DGARM; f.dq_rm = DQRM;
        f.de_out = x + W.DE; f.dconv_out = reinterpret_cast<uint16_t *>(x + W.DCONV); f.dctx_out = x + W.DCTX;
        f.dctxx = (unsigned long long *)(x + W.DCTXX); f.dqx = (unsigned long long *)(x + W.DQX);
        f.bar = (unsigned *)(x + W.BARA); f.err = err;
        f.drop = make_drop(seed, d.p_att, training);
        f.row_offset = row_offset; f.B = B; f.N = N; f.T = T; f.RS = fb_row_split(B, N);
        GVX_TRY(launch_att_chain_bwd(f, st));
    }
    pdl_barrier_next();
    for (int t = T - 1; t >= 0 && !fb; --t) {
        const bool last = t == T - 1;
        float *pdxd = x + W.PDXD + (size_t)(t & 1) * W.pdxd_stride, *pdxd_n = x + W.PDXD + (size_t)((t + 1) & 1) * W.pdxd_stride;
        float *pdxa = x + W.PDXA + (size_t)(t & 1) * W.pdxa_stride, *pdxa_n = x + W.PDXA + (size_t)((t + 1) & 1) * W.pdxa_stride;
        const long long sd = (long long)B * ldd, sa = (long long)B * lda;
        const float *dxd_t = x + W.DXDALL + (size_t)t * B * AE;
        if (!pc) {   // S1: decoder-LSTM pointwise backward
            ProfScope ps(PS_BWD_DEC_POINT, st);
            BfDsts dg;
            memset(&dg, 0, sizeof(dg));
            add_img(dg, GDI, 0, NPAD); add_rm(dg, DGDRM + (size_t)t * B * 4 * d.H, 0, 4 * d.H);
            GVX_TRY(run_bf_lstm_bwd(d, 1, src_plain(x + W.DHC + (size_t)t * B * d.Kp, d.Kp),
                                    last ? src_none() : src_split(pdxd_n + d.A + d.E, ldd, W.KSdT, sd), src_none(),
                                    s + S.GD + (size_t)t * 4 * BH, s + S.CD + t * BH, s + S.CD + (t + 1) * BH, x + W.DCD, dg, B, seed,
                                    t, training, row_offset, nullptr, nullptr, nullptr, st));
        }
        if (!pc) {   // S2: d x_dec = d gates_dec . W_dec
            ProfScope ps(PS_BWD_DEC_GEMM, st);
            GVX_TRY(run_tc(WdTI, GDI, pdxd, gm.TdT, gm.G4H, W.KSdT, B, err, st));
        }
        {   // S3: attention backward
            ProfScope ps(PS_BWD_ATTENTION, st);
            AttnBwdArgs a;
            memset(&a, 0, sizeof(a));
            a.s = AttnShape{B, N, d.D, d.E, d.F, d.KS};
            a.memory = memory; a.wlc = w->loc_conv_w; a.wld = w->loc_dense_w; a.v = w->v_w; a.lengths = mem_lengths;
            a.w_t = s + S.ALIGN + (size_t)t * N; a.w_bstride = (long long)T * N;
            a.th = s + S.TH + (size_t)t * B * N * d.D;
            a.dctx1 = src_plain(x + W.DHC + (size_t)t * B * d.Kp + d.H, d.Kp);
            a.dctx2 = pc ? src_plain(dxd_t + d.A, AE) : src_split(pdxd + d.A, ldd, W.KSdT, sd);
            a.dctx3 = last ? src_none() : src_split(pdxa_n + d.P, lda, W.KSaT, sa);
            a.d_align = d_align ? d_align + (size_t)t * N : nullptr; a.da_bstride = (long long)T * N;
            a.dw_carry = x + W.DW; a.dcum_carry = x + W.DCUM;
            a.dctx_out = x + W.DCTX + t * BE;
            a.de_out = x + W.DE + (size_t)t * B * N;
            a.dq_out = nullptr;
            add_img(a.dq_bf, DQI, 0, NPAD); add_rm(a.dq_bf, DQRM + (size_t)t * B * d.D, 0, d.D);
            a.dconv_out = x + W.DCONV + (size_t)t * B * N * d.F;
            a.dbg = pc_dbg_buffer() ? pc_dbg_buffer() + 32 * 1024 : nullptr;     // plane 1, row = frame (the decoder-LSTM BPTT chain
            a.dbg_t = t;                                                         // of the same call wrote its stamps there before)
            if (have_memb) a.memb = (const bf16 *)(s + S.MEMB);
            a.dctx12_static = pc ? 1 : 0;      // DHC and DXDALL are complete before the per-step chain starts
            if (dhq_folded) { a.WqB = (const bf16 *)(packed + BL.WqB); a.dhq_out = x + W.PS4; a.A = d.A; }
            GVX_TRY(launch_attention_bwd_best(a, st));
        }
        {   // S4: d h_att = d q . W_query + (from decoder-LSTM input) + (from step t+1), attention-LSTM pointwise backward
            ProfScope ps(PS_BWD_ATT_POINT, st);
            BfDsts dg;
            memset(&dg, 0, sizeof(dg));
            add_img(dg, GAI, 0, NPAD); add_rm(dg, DGARM + (size_t)t * B * 4 * d.A, 0, 4 * d.A);
            SrcSum dpre = last ? src_none() : src_split(pdxa_n, lda, W.KSaT, sa);
            const SrcSum s1 = pc ? src_plain(dxd_t, AE) : src_split(pdxd, ldd, W.KSdT, sd);
            const SrcSum s2 = last ? src_none() : src_split(pdxa_n + d.P + d.E, lda, W.KSaT, sa);
            if (s4_fused) {
                // d q . W_query inside the pointwise kernel: one launch instead of a K = 128 engine GEMM + pointwise
                GVX_TRY(run_bf_lstm_bwd_q(d, DQRM + (size_t)t * B * d.D, packed + PL.WqT, s1, s2, s + S.GA + (size_t)t * 4 * BA,
                                          s + S.CA + t * BA, s + S.CA + (t + 1) * BA, x + W.DCA, dg, B, seed, t, training, row_offset,
                                          last ? nullptr : &dpre, last ? nullptr : s + S.PRE2 + (size_t)(t + 1) * B * d.P,
                                          last ? nullptr : x + W.DZ2 + (size_t)(t + 1) * B * d.P, st));
            } else {
                if (!dhq_folded) GVX_TRY(run_tc(WqTI, DQI, x + W.PS4, gm.TqT, gm.Dp, W.KSs4, B, err, st));
                GVX_TRY(run_bf_lstm_bwd(d, 0, dhq_folded ? src_plain(x + W.PS4, d.A) : src_split(x + W.PS4, lds4, W.KSs4, (long long)B * lds4), s1, s2,
                                        s + S.GA + (size_t)t * 4 * BA, s + S.CA + t * BA, s + S.CA + (t + 1) * BA, x + W.DCA, dg, B, seed,
                                        t, training, row_offset, last ? nullptr : &dpre, last ? nullptr : s + S.PRE2 + (size_t)(t + 1) * B * d.P,
                                        last ? nullptr : x + W.DZ2 + (size_t)(t + 1) * B * d.P, st));
            }
        }
        {   // S5: d x_att = d gates_att . W_att
            ProfScope ps(PS_BWD_ATT_GEMM, st);
            GVX_TRY(run_tc(WaTI, GAI, pdxa, gm.TaT, gm.G4A, W.KSaT, B, err, st));
        }
    }
    ProfScope ps_batched(PS_BWD_BATCHED, st);
    if (fb) {   // prenet columns of d x_att for all frames: d gates_att . W_ih[:, prenet], then the relu / dropout mask (:143)
        if (own_gemm()) GVX_TRY(nt_gemm_bf16(st, TB, d.P, 4 * d.A, DGARM, 4 * d.A, (const bf16 *)(packed + BL.WaTRM), 4 * d.A, x + W.DZ1, d.P, err));
        else GVX_TRY(gemm_nn_bf16(st, TB, d.P, 4 * d.A, DGARM, 4 * d.A, (const bf16 *)(packed + BL.WaPRM), d.P, x + W.DZ1, d.P));
        k_prenet_bwd_mask<<<grid_for((size_t)TB * d.P), 256, 0, st>>>(x + W.DZ1, d.P, s + S.PRE2, TB, d.P, x + W.DZ2);
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
    } else {   // prenet gradient of frame 0 from the last d x_att partials (ping-pong half 0)
        const int total = B * d.P;
        BfLstmBwd a;
        memset(&a, 0, sizeof(a));
        a.main_blocks = 0; a.B = B; a.P = d.P;
        a.dpre_src = src_split(x + W.PDXA, lda, W.KSaT, (long long)B * lda);
        a.pre2 = s + S.PRE2; a.dz2 = x + W.DZ2;
        k_bf_lstm_bwd<<<grid_for((size_t)total), 256, 0, st>>>(a);
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
    }
    // projections: d Wpg = DOUT^T . [h_dec | ctx];  biases = column sums
    float *tmp = x + W.TMP;
    // weight gradients: d W = G^T . X over all frames.  Own GEMM: the frame-major operands are consumed as they lie in HBM (MN-major
    // tcgen05 operands, gvx_nt_gemm.cuh: no transpose pass), small outputs split over K (deterministic reduction)
    const bool og = own_gemm();
    if (og) GVX_TRY(tn_gemm_bf16(st, d.M + 1, d.Kp, TB, DOUTB, OLB, HCRM, d.Kp, tmp, d.Kp, err, x + W.GWS, W.gws_floats));
    else GVX_TRY(gemm_tn_bf16(st, d.M + 1, d.Kp, TB, DOUTB, OLB, HCRM, d.Kp, tmp, d.Kp));
    GVX_CUDA(cudaMemcpyAsync(g->proj_w, tmp, (size_t)d.M * d.Kp * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_CUDA(cudaMemcpyAsync(g->gate_w, tmp + (size_t)d.M * d.Kp, (size_t)d.Kp * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_TRY(colsum(st, x + W.DOUT, TB, d.M + 1, d.OL, x + W.ONES, x + W.DBIAS));
    GVX_CUDA(cudaMemcpyAsync(g->proj_b, x + W.DBIAS, (size_t)d.M * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_CUDA(cudaMemcpyAsync(g->gate_b, x + W.DBIAS + d.M, sizeof(float), cudaMemcpyDeviceToDevice, st));
    // LSTM weights (unit-major rows, [W_ih | W_hh] columns) and biases
    auto colsum_bf = [&](const bf16 *m, int cols, float *out) -> int {
        dim3 grid((cols + 255) / 256, W.colchunks);
        k_colsum_bf16_part<<<grid, 256, 0, st>>>(m, (size_t)TB, cols, W.colchunks, x + W.COLP);
        GVX_LAUNCHED(1);
        k_reduce_partials<<<(cols + 31) / 32, dim3(32, 8), 0, st>>>(x + W.COLP, W.colchunks, cols, 0, cols, out);
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
        return 0;
    };
    if (og) GVX_TRY(tn_gemm_bf16(st, 4 * d.H, d.Kd, TB, DGDRM, 4 * d.H, XDRM, d.Kd, x + W.DWD, d.Kd, err, x + W.GWS, W.gws_floats));
    else GVX_TRY(gemm_tn_bf16(st, 4 * d.H, d.Kd, TB, DGDRM, 4 * d.H, XDRM, d.Kd, x + W.DWD, d.Kd));
    k_unpack_lstm_grad<<<grid_for((size_t)4 * d.H * d.Kd), 256, 0, st>>>(x + W.DWD, d.H, d.A + d.E, g->dec_w_ih, g->dec_w_hh);
    GVX_LAUNCHED(1);
    GVX_TRY(colsum_bf(DGDRM, 4 * d.H, x + W.DBIAS));
    k_unpack_bias_grad<<<grid_for((size_t)4 * d.H), 256, 0, st>>>(x + W.DBIAS, d.H, g->dec_b_ih, g->dec_b_hh);
    GVX_LAUNCHED(1);
    if (og) GVX_TRY(tn_gemm_bf16(st, 4 * d.A, d.Ka, TB, DGARM, 4 * d.A, XARM, d.Ka, x + W.DWA, d.Ka, err, x + W.GWS, W.gws_floats));
    else GVX_TRY(gemm_tn_bf16(st, 4 * d.A, d.Ka, TB, DGARM, 4 * d.A, XARM, d.Ka, x + W.DWA, d.Ka));
    k_unpack_lstm_grad<<<grid_for((size_t)4 * d.A * d.Ka), 256, 0, st>>>(x + W.DWA, d.A, d.P + d.E, g->att_w_ih, g->att_w_hh);
    GVX_LAUNCHED(1);
    GVX_TRY(colsum_bf(DGARM, 4 * d.A, x + W.DBIAS));
    k_unpack_bias_grad<<<grid_for((size_t)4 * d.A), 256, 0, st>>>(x + W.DBIAS, d.A, g->att_b_ih, g->att_b_hh);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    // query layer: d Wq [D, A] = DQ^T . h_att   (h_att_t = first A columns of the decoder-LSTM input rows)
    if (og) GVX_TRY(tn_gemm_bf16(st, d.D, d.A, TB, DQRM, d.D, XDRM, d.Kd, g->query_w, d.A, err, x + W.GWS, W.gws_floats));
    else GVX_TRY(gemm_tn_bf16(st, d.D, d.A, TB, DQRM, d.D, XDRM, d.Kd, g->query_w, d.A));

    BwdPostArgs pa;
    pa.TH = s + S.TH; pa.DE = x + W.DE; pa.CONVS = s + S.CONVS; pa.DCONV = x + W.DCONV; pa.ALIGN = s + S.ALIGN;
    pa.CUMS = s + S.CUMS; pa.DCTX = x + W.DCTX; pa.PRE1 = s + S.PRE1; pa.FR = s + S.FR;
    pa.DPM = x + W.DPM; pa.PART1 = x + W.PART1; pa.PART2 = x + W.PART2; pa.DZ2 = x + W.DZ2; pa.DZ1 = x + W.DZ1;
    pa.post_blocks = W.post_blocks;
    pa.bf16_mode = 1;
    pa.th_bf16 = fb ? 1 : 0;
    GVX_TRY(bwd_post_common(d, w, memory, B, N, T, pa, g, d_memory, st));
    GVX_TRY(latch_record(err, 1, 2, st));
    GVX_LAUNCHED(1);
    return 0;
}

// ======================================================================================= inference
// One decoder step (tacotron2.py:398-403): prenet on the previous mel frame `prev` (straight into the attention-LSTM operand
// image), attention LSTM, query, attention (weights to align_t, row stride align_bstride), decoder LSTM, [mel | gate] projection
// to out_t.  row_frame / row_id: optional per-row prenet dropout frame and row (run_infer_prenet, run_prenet).
static int infer_step_bf16(const Dims &d, const gvx_weights *w, const float *packed, const InferBfL &L, float *s, const float *memory,
                           const int64_t *mem_lengths, int B, int N, uint64_t seed, int t, int training, int row_offset,
                           const int *row_frame, const int *row_id, const float *prev, float *align_t, long long align_bstride,
                           float *out_t, cudaStream_t st) {
    const BfGeom g(d);
    const PackedL PL(d);
    const PackedBfL BL(d, PL.total);
    const int NPAD = L.NPAD;
    bf16 *XAI = (bf16 *)(s + L.XAI), *XDI = (bf16 *)(s + L.XDI), *XPI = (bf16 *)(s + L.XPI);
    int *err = (int *)(s + L.ERR), *flags = (int *)(s + L.FLAGS);
    const bf16 *WaI = (const bf16 *)(packed + BL.WaI), *WdI = (const bf16 *)(packed + BL.WdI), *WqI = (const bf16 *)(packed + BL.WqI),
               *WpgI = (const bf16 *)(packed + BL.WpgI);
    bf16 *xa = XAI + (size_t)(t & 1) * L.xai_stride, *xa_n = XAI + (size_t)((t + 1) & 1) * L.xai_stride;
    bf16 *xd = XDI + (size_t)(t & 1) * L.xdi_stride, *xd_n = XDI + (size_t)((t + 1) & 1) * L.xdi_stride;
    {
        ProfScope ps(PS_PRENET, st);
        BfDsts bf;
        memset(&bf, 0, sizeof(bf));
        add_img(bf, xa, 0, NPAD);
        if (infer_prenet_fused_ok(d, B)) {
            GVX_TRY(run_infer_prenet(d, w, prev, d.OL, B, seed, t, row_offset, s + L.PRE1, nullptr, &bf, (unsigned *)(flags + 40), err, st,
                                     row_frame, row_id));
        } else {
            GVX_TRY(run_prenet(d, w, prev, d.OL, B, B, seed, t, row_offset, s + L.PRE1, s + L.PRE2, st, &bf, row_frame, row_id));
        }
    }
    {
        ProfScope ps(PS_ATT_LSTM, st);
        BfDsts h;
        memset(&h, 0, sizeof(h));
        add_img(h, xd, 0, NPAD); add_img(h, xa_n, d.P + d.E, NPAD);
        GVX_TRY(run_lstm_bf16(d, packed, 0, WaI, xa, s + L.PA, L.KSa, g.Ta, g.Kpa, s + L.CA, s + L.CA, nullptr, h, B, seed, t,
                              training, row_offset, err, st));
    }
    {
        ProfScope ps(PS_QUERY, st);
        GVX_TRY(run_tc(WqI, xd, s + L.PQ, g.Tq, g.Kpq, L.KSq, B, err, st));
    }
    {
        ProfScope ps(PS_ATTENTION, st);
        AttnFwdArgs a;
        memset(&a, 0, sizeof(a));
        a.s = AttnShape{B, N, d.D, d.E, d.F, d.KS};
        a.q = src_split(s + L.PQ, g.Tq * TC_M, L.KSq, (long long)B * g.Tq * TC_M);
        a.pm = s + L.PM; a.memory = memory;
        a.wlc = w->loc_conv_w; a.wldT = packed + PL.wldT; a.v = w->v_w; a.lengths = mem_lengths;
        a.w_prev = s + L.WPREV; a.cum = s + L.CUM;
        a.align_out = align_t; a.align_bstride = align_bstride;
        a.ctx_ld = d.E;
        add_img(a.ctx_bf, xd, d.A, NPAD); add_img(a.ctx_bf, xa_n, d.P, NPAD); add_img(a.ctx_bf, XPI, d.H, NPAD);
        GVX_TRY(launch_attention_fwd_best(a, st));
    }
    {
        ProfScope ps(PS_DEC_LSTM, st);
        BfDsts h;
        memset(&h, 0, sizeof(h));
        add_img(h, XPI, 0, NPAD); add_img(h, xd_n, d.A + d.E, NPAD);
        GVX_TRY(run_lstm_bf16(d, packed, 1, WdI, xd, s + L.PD, L.KSd, g.Td, g.Kpd, s + L.CD, s + L.CD, nullptr, h, B, seed, t,
                              training, row_offset, err, st));
    }
    {
        ProfScope ps(PS_PROJ, st);
        GVX_TRY(run_tc(WpgI, XPI, s + L.PP, g.Tp, g.Kpp, L.KSp, B, err, st));
        GVX_CUDA(launch_pdl(k_bf_finalize, dim3(grid_for((size_t)B * (d.M + 1))), dim3(256), 0, st, (const float *)(s + L.PP), L.KSp,
                            B, g.Tp * TC_M, d.M + 1, (const float *)(packed + PL.bpg), out_t, d.OL));
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
    }
    return 0;
}

int infer_bf16(const Dims &d, const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths,
                      int B, int N, int max_steps, float gate_threshold, int ignore_gate, uint64_t seed, int training,
                      int row_offset, float *mel_out, float *gate_out, float *align_out, int32_t *n_frames, int *steps_run, float *s,
                      cudaStream_t st) {
    GVX_TRY(check_bf16_dims(d, B));
    const BfGeom g(d);
    const InferBfL L(d, B, N, max_steps);
    const int NPAD = L.NPAD;
    bf16 *XAI = (bf16 *)(s + L.XAI), *XDI = (bf16 *)(s + L.XDI), *XPI = (bf16 *)(s + L.XPI);
    int *err = (int *)(s + L.ERR), *flags = (int *)(s + L.FLAGS);

    GVX_TRY(run_processed_memory(d, w, memory, B, N, s + L.PM, st));
    GVX_CUDA(cudaMemsetAsync(err, 0, 64 * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(flags, 0, 32 * sizeof(int), st));       // [0] rows still running; [32..33] hold the dropout seed (gvx_dec_infer)
    GVX_CUDA(cudaMemsetAsync(flags + 40, 0, 2 * sizeof(int), st));   // [40] prenet grid barrier
    GVX_CUDA(cudaMemsetAsync(XAI, 0, 2 * L.xai_stride * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(XDI, 0, 2 * L.xdi_stride * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(XPI, 0, (size_t)g.Kpp * NPAD * sizeof(bf16), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CA, 0, (size_t)B * d.A * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CD, 0, (size_t)B * d.H * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.WPREV, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CUM, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.ZERO, 0, (size_t)B * d.OL * sizeof(float), st));
    k_fill_i32<<<grid_for(B), 256, 0, st>>>(n_frames, B, ignore_gate ? max_steps : -1, 0);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());

    int t = 0, host_running = B;
    pdl_barrier_next();
    for (; t < max_steps; ++t) {
        const float *prev = t == 0 ? s + L.ZERO : s + L.OUT + (size_t)(t - 1) * B * d.OL;
        float *out_t = s + L.OUT + (size_t)t * B * d.OL;
        GVX_TRY(infer_step_bf16(d, w, packed, L, s, memory, mem_lengths, B, N, seed, t, training, row_offset, nullptr, nullptr, prev,
                                align_out + (size_t)t * N, (long long)max_steps * N, out_t, st));
        if (!ignore_gate) {
            GVX_CUDA(launch_pdl(k_gate_check, dim3(1), dim3(128), 0, st, (const float *)out_t, B, d.M, d.OL, gate_threshold, t, n_frames, flags));
            GVX_LAUNCHED(1);
            GVX_CUDA(cudaGetLastError());
            if ((t + 1) % GVX_STOP_POLL == 0 || t + 1 == max_steps) {
                GVX_CUDA(cudaMemcpyAsync(&host_running, flags, sizeof(int), cudaMemcpyDeviceToHost, st));
                GVX_CUDA(cudaStreamSynchronize(st));
                if (host_running == 0) { ++t; break; }
            }
        }
    }
    const int steps = t < max_steps ? t : max_steps;
    if (!ignore_gate) {
        k_fill_i32<<<grid_for(B), 256, 0, st>>>(n_frames, B, steps, 1);
        GVX_LAUNCHED(1);
    }
    k_unpack_out<<<grid_for((size_t)B * (d.M + 1) * steps), 256, 0, st>>>(s + L.OUT, B, d.M, d.OL, steps, max_steps, mel_out, gate_out);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    *steps_run = steps;
    return 0;
}

size_t packed_total_bf16(const Dims &d) { return PackedBfL(d, PackedL(d).total).total; }
size_t stash_total_bf16(const Dims &d, int B, int N, int T) { return StashBfL(d, B, N, T).total; }
size_t bwd_total_bf16(const Dims &d, int B, int N, int T) { return BwdBfL(d, B, N, T).total; }
size_t infer_total_bf16(const Dims &d, int B, int N, int steps) { return InferBfL(d, B, N, steps).total; }
size_t stash_seed_off_bf16(const Dims &d, int B, int N, int T) { return StashBfL(d, B, N, T).SEED; }
size_t infer_flags_off_bf16(const Dims &d, int B, int N, int steps) { return InferBfL(d, B, N, steps).FLAGS; }
size_t infer_err_off_bf16(const Dims &d, int B, int N, int steps) { return InferBfL(d, B, N, steps).ERR; }
int check_tc_err_public(int *err_dev, cudaStream_t st, const char *what) { return check_tc_err(err_dev, st, what); }

}  // namespace gvx

// ---- debug hook: device buffer ([4][1024][32] long long: decoder-LSTM forward chain, backward chain, progress markers, fused attention chain) receiving clock64 stamps of CTA 0
// ---- debug hook: force a code path on (1) / off (0) / back to the environment default (-1)
extern "C" int gvx_debug_option(const char *name, int value) {
    if (!strcmp(name, "fused")) gvx::fa_mode() = value;
    else if (!strcmp(name, "persistent")) gvx::pc_mode() = value;
    else { snprintf(gvx::g_err, sizeof(gvx::g_err), "gvx_debug_option: unknown option %s", name); return 1; }
    return 0;
}

extern "C" int gvx_debug_timeline(void *device_buffer) {
    gvx::pc_dbg_buffer() = (long long *)device_buffer;
    return 0;
}

// ---- test hook: the own tcgen05 GEMM on its own: C[M,N] = A[M,K] . B[N,K]^T (mode 0, K-major operands), or with mode 1 A given as
// [K,M] and B as [K,N] (MN-major operands, the weight-gradient path).  fp32 in, rounded to bf16 on the device.
extern "C" int gvx_test_nt_gemm(const float *A, const float *B, int M, int N, int K, int mode, float *C, void *stream) {
    using namespace gvx;
    GVX_CHECK(A && B && C && M > 0 && N > 0 && K > 0 && K % 8 == 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    bf16 *a = nullptr, *b = nullptr, *at = nullptr, *bt = nullptr;
    int *err = nullptr;
    float *ws = nullptr;
    const size_t ws_floats = (size_t)32 << 20;           // the production workspace size: split-K is taken exactly as in training
    GVX_CUDA(cudaMalloc(&a, (size_t)M * K * 2));
    GVX_CUDA(cudaMalloc(&b, (size_t)N * K * 2));
    GVX_CUDA(cudaMalloc(&err, 64));
    GVX_CUDA(cudaMalloc(&ws, ws_floats * 4));
    GVX_CUDA(cudaMemsetAsync(err, 0, 64, st));
    int rc = 0;
    if (mode == 0) {
        k_to_bf16<<<grid_for((size_t)M * K), 256, 0, st>>>(A, K, (size_t)M, K, a, K);
        k_to_bf16<<<grid_for((size_t)N * K), 256, 0, st>>>(B, K, (size_t)N, K, b, K);
        rc = nt_gemm_bf16(st, M, N, K, a, K, b, K, C, N, err, ws, ws_floats);
    } else {
        GVX_CHECK(M % 8 == 0 && N % 8 == 0, "mode 1 needs M, N multiples of 8");
        k_to_bf16<<<grid_for((size_t)M * K), 256, 0, st>>>(A, M, (size_t)K, M, a, M);        // A given as [K, M]
        k_to_bf16<<<grid_for((size_t)N * K), 256, 0, st>>>(B, N, (size_t)K, N, b, N);        // B given as [K, N]
        rc = tn_gemm_bf16(st, M, N, K, a, M, b, N, C, N, err, ws, ws_floats);             // MN-major operands straight from memory
    }
    if (!rc) rc = check_tc_err(err, st, "nt_gemm");
    else cudaStreamSynchronize(st);
    cudaFree(a); cudaFree(b); cudaFree(at); cudaFree(bt); cudaFree(err); cudaFree(ws);
    return rc;
}

// ---- timing hook for profiles/nt_gemm_bench.py: average device time of `reps` launches on zero-filled operands
extern "C" int gvx_bench_nt_gemm(int M, int N, int K, int reps, float *ms_out) {
    using namespace gvx;
    bf16 *a = nullptr, *b = nullptr;
    float *c = nullptr, *ws = nullptr;
    int *err = nullptr;
    const size_t ws_floats = (size_t)32 << 20;
    GVX_CUDA(cudaMalloc(&ws, ws_floats * 4));
    GVX_CUDA(cudaMalloc(&a, (size_t)M * K * 2));
    GVX_CUDA(cudaMalloc(&b, (size_t)N * K * 2));
    GVX_CUDA(cudaMalloc(&c, (size_t)M * N * 4));
    GVX_CUDA(cudaMalloc(&err, 64));
    GVX_CUDA(cudaMemset(a, 0, (size_t)M * K * 2));
    GVX_CUDA(cudaMemset(b, 0, (size_t)N * K * 2));
    GVX_CUDA(cudaMemset(err, 0, 64));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    int rc = nt_gemm_bf16(0, M, N, K, a, K, b, K, c, N, err, ws, ws_floats);
    cudaEventRecord(e0, 0);
    for (int i = 0; i < reps && !rc; ++i) rc = nt_gemm_bf16(0, M, N, K, a, K, b, K, c, N, err, ws, ws_floats);
    cudaEventRecord(e1, 0);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    *ms_out = ms / (reps > 0 ? reps : 1);
    if (!rc) rc = check_tc_err(err, 0, "nt_gemm bench");
    cudaFree(a); cudaFree(b); cudaFree(c); cudaFree(err); cudaFree(ws);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

// ---- test hook: the persistent LSTM chain on its own (forward, then optionally BPTT) -----------------------------
__global__ void k_bf16_rows_to_f32(const __nv_bfloat16 *__restrict__ x, size_t n, float *__restrict__ y) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) y[i] = __bfloat162float(x[i]);
}

extern "C" int gvx_test_lstm_chain(const float *w_hh, const float *pre, int B, int T, int H, float p_drop, uint64_t seed,
                                   int training, float *h_out, float *c_out, float *gates_out, const float *dh_ext,
                                   float *dgates_out, void *stream) {
    using namespace gvx;
    GVX_CHECK(w_hh && pre && h_out && c_out && gates_out && B > 0 && T > 0, "bad argument");
    GVX_CHECK(pc_supported(H, B), "persistent chain: unsupported shape (need H % 64 == 0, H/8 <= SM count, B <= 64)");
    cudaStream_t st = (cudaStream_t)stream;
    bf16 *wimg = nullptr, *wimgT = nullptr, *himg = nullptr, *hrm = nullptr, *gimg = nullptr, *dgrm = nullptr;
    unsigned *bar = nullptr;
    int *err = nullptr;
    const size_t TBH = (size_t)T * B * H;
    GVX_CUDA(cudaMalloc(&wimg, pc_wimg_elems(H) * 2));
    GVX_CUDA(cudaMalloc(&wimgT, pc_wimg_elems(H) * 2));
    GVX_CUDA(cudaMalloc(&himg, pc_himg_elems(H) * 2));
    GVX_CUDA(cudaMalloc(&hrm, TBH * 2));
    GVX_CUDA(cudaMalloc(&gimg, pc_gimg_elems(H) * 2));
    GVX_CUDA(cudaMalloc(&dgrm, 4 * TBH * 2));
    GVX_CUDA(cudaMalloc(&bar, 256));
    GVX_CUDA(cudaMalloc(&err, 64));
    GVX_CUDA(cudaMemsetAsync(err, 0, 64, st));
    GVX_CUDA(cudaMemsetAsync(himg, 0, pc_himg_elems(H) * 2, st));
    GVX_CUDA(cudaMemsetAsync(gimg, 0, pc_gimg_elems(H) * 2, st));
    GVX_CUDA(cudaMemsetAsync(c_out, 0, (size_t)B * H * sizeof(float), st));
    k_pc_pack_w<<<grid_for(pc_wimg_elems(H)), 256, 0, st>>>(w_hh, H, H, 0, wimg);
    k_pc_pack_w<<<grid_for(pc_wimg_elems(H)), 256, 0, st>>>(w_hh, H, H, 1, wimgT);
    PcFwdArgs f;
    memset(&f, 0, sizeof(f));
    f.Wimg = wimg; f.pre = pre; f.himg = himg; f.c_stash = c_out; f.gates_stash = gates_out;
    f.out[0] = PcOut{hrm, H, 0, 0, (long long)B * H};
    f.bar = bar; f.err = err;
    f.drop = make_drop(seed, p_drop, training, nullptr);
    f.drop.kptr = nullptr;
    f.site = SITE_DEC; f.row_offset = 0; f.B = B; f.T = T; f.H = H;
    int rc = launch_lstm_chain_fwd(f, st);
    if (!rc) {
        k_bf16_rows_to_f32<<<grid_for(TBH), 256, 0, st>>>(hrm, TBH, h_out);
        if (dh_ext && dgates_out) {
            PcBwdArgs g;
            memset(&g, 0, sizeof(g));
            g.Wimg = wimgT; g.gimg = gimg; g.dh_ext = dh_ext; g.dh_ld = H; g.dh_tstride = (long long)B * H;
            g.gates_stash = gates_out; g.c_stash = c_out; g.dg_rm = dgrm; g.bar = bar; g.err = err;
            g.drop = f.drop; g.site = SITE_DEC; g.row_offset = 0; g.B = B; g.T = T; g.H = H;
            rc = launch_lstm_chain_bwd(g, st);
            if (!rc) k_bf16_rows_to_f32<<<grid_for(4 * TBH), 256, 0, st>>>(dgrm, 4 * TBH, dgates_out);
        }
    }
    if (!rc) rc = check_tc_err(err, st, "persistent lstm chain");
    else cudaStreamSynchronize(st);
    cudaFree(wimg); cudaFree(wimgT); cudaFree(himg); cudaFree(hrm); cudaFree(gimg); cudaFree(dgrm); cudaFree(bar); cudaFree(err);
    return rc;
}
