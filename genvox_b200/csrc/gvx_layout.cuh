// genvox_b200 — HBM layouts: packed weights, training stash, backward / inference workspaces.
// All offsets are in floats from the start of the caller-allocated buffer; every block is
// aligned to 64 floats (256 B) so any row start that is a multiple of 4 floats is 16-byte aligned.
#pragma once
#include "../../include/genvox_b200.h"
#include <stddef.h>

namespace gvx {

struct Dims {
    int M, E, A, H, P, D, F, KS;     // n_mels, enc, att_rnn, dec_rnn, prenet, att_dim, filters, kernel
    int Ka, Kd, Kp;                  // att-LSTM K = P+E+A, dec-LSTM K = A+E+H, projection K = H+E
    int OL;                          // row stride of the [mel | gate] output rows: round_up(M+1, 4)
    float p_att, p_dec;
    explicit Dims(const gvx_dims &d)
        : M(d.n_mels), E(d.enc_dim), A(d.att_rnn_dim), H(d.dec_rnn_dim), P(d.prenet_dim), D(d.att_dim),
          F(d.loc_filters), KS(d.loc_kernel), Ka(P + E + A), Kd(A + E + H), Kp(H + E), OL((M + 1 + 3) & ~3),
          p_att(d.p_att_dropout), p_dec(d.p_dec_dropout) {}
};

struct Carver {
    size_t o = 0;
    size_t take(size_t n) { size_t r = o; o += (n + 63) & ~(size_t)63; return r; }
};

// ---- packed weights --------------------------------------------------------------------------
// Wa  [4A, Ka]  attention_rnn: row 4*u+g <- torch row g*A+u, columns [W_ih | W_hh]; ba = b_ih + b_hh
// WaT [Ka, 4A]  transpose (backward dX GEMM wants K-major over the gate axis)
// Wd, bd, WdT   decoder_rnn, same scheme
// Wpg [M+1, Kp] linear_projection rows then the gate_layer row; bpg [M+1]
// WqT [A, D]    query_layer weight transposed;  wldT [F, D] location_dense weight transposed
struct PackedL {
    size_t Wa, ba, WaT, Wd, bd, WdT, Wpg, bpg, WqT, wldT, total;
    explicit PackedL(const Dims &d) {
        Carver c;
        Wa = c.take((size_t)4 * d.A * d.Ka); ba = c.take(4 * d.A); WaT = c.take((size_t)4 * d.A * d.Ka);
        Wd = c.take((size_t)4 * d.H * d.Kd); bd = c.take(4 * d.H); WdT = c.take((size_t)4 * d.H * d.Kd);
        Wpg = c.take((size_t)(d.M + 1) * d.Kp); bpg = c.take(d.M + 1);
        WqT = c.take((size_t)d.A * d.D); wldT = c.take((size_t)d.F * d.D);
        total = c.o;
    }
};

// ---- training stash (written by train_fwd, read by train_bwd); time-major [T][B][feat] ----------
struct StashL {
    size_t FR, PRE1, PRE2, PM, HA, CA, GA, CTX, HD, CD, GD, Q, ALIGN, CUMS, TH, CONVS, OUT, WPREV, CUM, SEED, total;
    StashL(const Dims &d, int B, int N, int T) {
        Carver c;
        const size_t TB = (size_t)T * B, T1B = (size_t)(T + 1) * B;
        FR = c.take(TB * d.M); PRE1 = c.take(TB * d.P); PRE2 = c.take(TB * d.P);
        PM = c.take((size_t)B * N * d.D);
        HA = c.take(T1B * d.A); CA = c.take(T1B * d.A); GA = c.take(TB * 4 * d.A);
        CTX = c.take(T1B * d.E);
        HD = c.take(T1B * d.H); CD = c.take(T1B * d.H); GD = c.take(TB * 4 * d.H);
        Q = c.take(TB * d.D);
        ALIGN = c.take((size_t)B * T * N); CUMS = c.take((size_t)B * T * N);
        TH = c.take(TB * N * d.D);           // [T][B][N][D] tanh(q + loc + pm)
        CONVS = c.take(TB * N * d.F);        // [T][B][N][F] location-conv output
        OUT = c.take(TB * d.OL);
        WPREV = c.take((size_t)B * N); CUM = c.take((size_t)B * N);
        SEED = c.take(64);                   // dropout seed of the call {lo, hi}, read by the kernels (graph replay)
        total = c.o;
    }
};

// ---- backward workspace -------------------------------------------------------------------------
struct BwdL {
    size_t DOUT, DHC, DGD, DGA, DXD, DXA, DCD, DCA, DCTX, DQ, DE, DCONV, DZ2, DZ1, DPM, DW, DCUM, DWA, DWD, DBIAS,
        PART1, PART2, ONES, TMP, total;
    int post_blocks;
    BwdL(const Dims &d, int B, int N, int T) {
        Carver c;
        const size_t TB = (size_t)T * B;
        post_blocks = 148 * 8;
        DOUT = c.take(TB * d.OL);            // [T][B][OL]   d(mel|gate) time-major
        DHC = c.take(TB * d.Kp);             // [T][B][H+E]  DOUT . Wpg
        DGD = c.take(TB * 4 * d.H);          // d(pre-activations) decoder LSTM, packed gate order
        DGA = c.take(TB * 4 * d.A);
        DXD = c.take((size_t)2 * B * d.Kd);  // per-step d(x_dec) = [d h_att | d ctx | d h_dec(prev)], ping-pong
        DXA = c.take(TB * d.Ka);             // [T][B][Ka] d(x_att) = [d prenet_out | d ctx(prev) | d h_att(prev)]
        DCD = c.take((size_t)B * d.H);       // carried d(c)
        DCA = c.take((size_t)B * d.A);
        DCTX = c.take(TB * d.E);             // total d(ctx_t)
        DQ = c.take(TB * d.D);
        DE = c.take(TB * N);                 // [T][B][N] d energies
        DCONV = c.take(TB * N * d.F);        // [T][B][N][F]
        DZ2 = c.take(TB * d.P);
        DZ1 = c.take(TB * d.P);
        DPM = c.take((size_t)B * N * d.D);
        DW = c.take((size_t)B * N);
        DCUM = c.take((size_t)B * N);
        DWA = c.take((size_t)4 * d.A * d.Ka);   // packed-layout weight grads
        DWD = c.take((size_t)4 * d.H * d.Kd);
        DBIAS = c.take((size_t)4 * (d.A > d.H ? d.A : d.H));
        PART1 = c.take((size_t)post_blocks * (d.D * d.F + d.D));     // per-block partials: d Wld, d v
        PART2 = c.take((size_t)post_blocks * d.F * 2 * d.KS);        // per-block partials: d Wlc
        ONES = c.take(TB);
        TMP = c.take((size_t)(d.M + 1) * d.Kp + 64);
        total = c.o;
    }
};

// ---- inference workspace --------------------------------------------------------------------------
struct InferL {
    size_t PM, PRE1, PRE2, HA, CA, CTX, HD, CD, Q, WPREV, CUM, OUT, ZERO, FLAGS, total;
    InferL(const Dims &d, int B, int N, int steps) {
        Carver c;
        PM = c.take((size_t)B * N * d.D);
        PRE1 = c.take((size_t)B * d.P); PRE2 = c.take((size_t)B * d.P);
        HA = c.take((size_t)2 * B * d.A); CA = c.take((size_t)B * d.A);
        CTX = c.take((size_t)B * d.E);
        HD = c.take((size_t)2 * B * d.H); CD = c.take((size_t)B * d.H);
        Q = c.take((size_t)B * d.D);
        WPREV = c.take((size_t)B * N); CUM = c.take((size_t)B * N);
        OUT = c.take((size_t)steps * B * d.OL);
        ZERO = c.take((size_t)B * d.OL);     // the all-zero go frame (tacotron2.py:392)
        FLAGS = c.take(64);
        total = c.o;
    }
};

// per-step arguments of the inference step functions (infer_step, infer_step_bf16)
struct InferStepArgs {
    const float *memory;
    const int64_t *lengths;
    const int *row_frame, *row_id;     // optional per-row prenet dropout frame and row (run_prenet), or null
    const float *prev;                 // the previous [mel | gate] rows (the go frame at the first step)
    float *align_t;                    // this step's attention weights, row stride align_bstride
    long long align_bstride;
    float *out_t;                      // this step's [mel | gate] rows
    int t;
    uint64_t seed;
    int training, row_offset;
    int win_back, win_fwd;             // the attention constraint (AttnFwdArgs; win_fwd == 0: off)
};

}  // namespace gvx
