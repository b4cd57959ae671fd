// genvox_b200 — C-ABI entry points: weight repack, teacher-forced forward, batched inference,
// and the single-phase hooks used by the parity tests.  See include/genvox_b200.h for the
// contract and the reference file:line each entry point replaces.
#include "../../include/genvox_b200.h"
#include "gvx_infer_prenet.cuh"
#include "gvx_attention_c2.cuh"
#include "gvx_common.cuh"
#include "gvx_gemm.cuh"
#include "gvx_graph.cuh"
#include "gvx_layout.cuh"
#include "gvx_misc.cuh"
#include "gvx_tc.cuh"
#include "gvx_bf16.cuh"
#include "gvx_blas.cuh"

namespace gvx {
thread_local char g_err[512] = {0};

// bf16 mode drivers (gvx_bf16_api.cuh, same translation unit)
size_t packed_total_bf16(const Dims &d);
size_t stash_total_bf16(const Dims &d, int B, int N, int T);
size_t bwd_total_bf16(const Dims &d, int B, int N, int T);
size_t infer_total_bf16(const Dims &d, int B, int N, int steps);
size_t stash_seed_off_bf16(const Dims &d, int B, int N, int T);
size_t infer_flags_off_bf16(const Dims &d, int B, int N, int steps);
size_t infer_err_off_bf16(const Dims &d, int B, int N, int steps);
int check_tc_err_public(int *err_dev, cudaStream_t st, const char *what);
int pack_weights_bf16(const Dims &d, const gvx_weights *w, float *packed, cudaStream_t st);
int train_fwd_bf16(const Dims &d, const gvx_weights *w, const float *packed, const float *memory, const float *mel_in,
                   const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training, int row_offset, float *mel_out,
                   float *gate_out, float *align_out, float *s, cudaStream_t st);
int infer_bf16(const Dims &d, const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths, int B,
               int N, int max_steps, float gate_threshold, int ignore_gate, uint64_t seed, int training, int row_offset,
               float *mel_out, float *gate_out, float *align_out, int32_t *n_frames, int *steps_run, float *s, cudaStream_t st);

int check_dims(const gvx_dims *d) {
    GVX_CHECK(d != nullptr, "dims is null");
    GVX_CHECK(d->n_mels > 0 && d->enc_dim > 0 && d->att_rnn_dim > 0 && d->dec_rnn_dim > 0 && d->prenet_dim > 0 &&
                  d->att_dim > 0 && d->loc_filters > 0 && d->loc_kernel > 0,
              "all dims must be positive");
    GVX_CHECK(d->n_mels % 4 == 0 && d->enc_dim % 4 == 0 && d->att_rnn_dim % 4 == 0 && d->dec_rnn_dim % 4 == 0 &&
                  d->prenet_dim % 4 == 0 && d->att_dim % 4 == 0,
              "n_mels, enc_dim, rnn dims, prenet_dim and att_dim must be multiples of 4");
    GVX_CHECK(d->loc_kernel % 2 == 1, "attention_location_kernel_size must be odd");
    GVX_CHECK(d->p_att_dropout >= 0.f && d->p_att_dropout < 1.f && d->p_dec_dropout >= 0.f && d->p_dec_dropout < 1.f,
              "dropout probabilities must be in [0, 1)");
    GVX_CHECK(d->precision == GVX_FP32 || d->precision == GVX_BF16, "precision must be GVX_FP32 or GVX_BF16");
    if (d->precision == GVX_BF16)
        GVX_CHECK(d->n_mels % 8 == 0 && d->enc_dim % 8 == 0 && d->att_rnn_dim % 32 == 0 && d->dec_rnn_dim % 32 == 0 &&
                      d->prenet_dim % 8 == 0 && d->att_dim % 8 == 0,
                  "bf16 mode: feature dims must be multiples of 8 and the rnn dims multiples of 32");
    return 0;
}

// ReLU + always-on dropout of a prenet layer in place (tacotron2.py:143), plus the optional bf16 copies: the epilogue of the
// time-batched path below.  Element (row m, column c): frame m / rows_per_frame, batch row m % rows_per_frame.
__global__ void __launch_bounds__(256) k_prenet_epilogue(float *__restrict__ x, int ld, size_t rows, int cols, DropCfg drop, uint32_t site,
                                                         int t0, int rows_per_frame, int row_offset, BfDsts bf,
                                                         const int *__restrict__ row_frame, const int *__restrict__ row_id) {
    const size_t total = rows * (size_t)cols;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t m = i / cols;
        const int c = (int)(i - m * cols);
        const int f = (int)(m / rows_per_frame), brow = (int)(m - (size_t)f * rows_per_frame);
        const uint32_t tf = row_frame ? (uint32_t)row_frame[brow] : (uint32_t)(t0 + f);
        const uint32_t rw = (uint32_t)((row_id ? row_id[brow] : brow) + row_offset);
        const float v = fmaxf(x[m * ld + c], 0.f) * drop_mult(drop, site, tf, rw, (uint32_t)c);
        x[m * ld + c] = v;
        if (bf.n) bf_store1_t(bf, f, brow, c, v);
    }
}

// Prenet.forward over `rows` = F*B rows (tacotron2.py:140-144).  row_frame / row_id (optional, device [B], one frame only):
// per-row Philox t and row (before row_offset) in place of t0 and the batch row.
int run_prenet(const Dims &d, const gvx_weights *w, const float *frames, int frames_ld, int rows, int B, uint64_t seed,
               int t0, int row_offset, float *pre1, float *pre2, cudaStream_t st, const BfDsts *bf = nullptr,
               const int *row_frame = nullptr, const int *row_id = nullptr) {
    if (rows >= 4096) {
        // all frames of a teacher-forced pass at once: a plain fp32 library GEMM per layer (exact fp32 products, like the skinny
        // FFMA kernel below, which needs 0.84 ms for the 51200 rows of configs[2]) + one elementwise pass
        for (int layer = 0; layer < 2; ++layer) {
            float *out = layer == 0 ? pre1 : pre2;
            if (layer == 0) GVX_TRY(sgemm_nt(st, rows, d.P, d.M, frames, frames_ld, w->prenet_w0, d.M, out, d.P));
            else GVX_TRY(sgemm_nt(st, rows, d.P, d.P, pre1, d.P, w->prenet_w1, d.P, out, d.P));
            BfDsts none;
            memset(&none, 0, sizeof(none));
            k_prenet_epilogue<<<grid_for((size_t)rows * d.P), 256, 0, st>>>(out, d.P, (size_t)rows, d.P, make_drop(seed, 0.5f, 1),
                                                                          layer == 0 ? SITE_PRENET0 : SITE_PRENET1, t0, B, row_offset,
                                                                          (layer == 1 && bf) ? *bf : none, row_frame, row_id);
            GVX_LAUNCHED(1);
            GVX_CUDA(cudaGetLastError());
        }
        return 0;
    }
    for (int layer = 0; layer < 2; ++layer) {
        GemmIn g = gemm_in(layer == 0 ? w->prenet_w0 : w->prenet_w1, layer == 0 ? d.M : d.P, d.P, rows);
        if (layer == 0) add_seg(g, frames, d.M, frames_ld);
        else add_seg(g, pre1, d.P, d.P);
        EpiStore e;
        memset(&e, 0, sizeof(e));
        e.out = layer == 0 ? pre1 : pre2;
        e.ldo = d.P;
        e.mode = 1;
        e.drop = make_drop(seed, 0.5f, 1);
        e.site = layer == 0 ? SITE_PRENET0 : SITE_PRENET1;
        e.t0 = t0;
        e.rows_per_frame = B;
        e.row_offset = row_offset;
        e.row_frame = row_frame;
        e.row_id = row_id;
        if (layer == 1 && bf) e.bf = *bf;
        GVX_TRY((launch_gemm<32, EpiStore>(g, e, st)));
    }
    return 0;
}

// processed_memory = memory_layer(memory)  (tacotron2.py:314)
int run_processed_memory(const Dims &d, const gvx_weights *w, const float *memory, int B, int N, float *pm, cudaStream_t st) {
    GemmIn g = gemm_in(w->memory_w, d.E, d.D, B * N);
    add_seg(g, memory, d.E, d.E);
    EpiStore e;
    memset(&e, 0, sizeof(e));
    e.out = pm;
    e.ldo = d.D;
    return launch_gemm<32, EpiStore>(g, e, st);
}

struct LstmIO {
    const float *x0; int w0, ld0;
    const float *x1; int w1, ld1;
    const float *x2; int w2, ld2;
    const float *c_prev;
    float *c_out, *h_out, *gates_out;
};

int run_lstm(const Dims &d, const float *packed, int which, const LstmIO &io, int B, uint64_t seed, int t, int training,
             int row_offset, cudaStream_t st) {
    const PackedL PL(d);
    const int HID = which == 0 ? d.A : d.H, K = which == 0 ? d.Ka : d.Kd;
    GemmIn g = gemm_in(packed + (which == 0 ? PL.Wa : PL.Wd), K, 4 * HID, B);
    add_seg(g, io.x0, io.w0, io.ld0);
    if (io.x1) add_seg(g, io.x1, io.w1, io.ld1);
    if (io.x2) add_seg(g, io.x2, io.w2, io.ld2);
    GVX_CHECK(io.w0 + io.w1 + io.w2 == K, "LSTM input widths do not add up");
    EpiLstm e;
    memset(&e, 0, sizeof(e));
    e.bias = packed + (which == 0 ? PL.ba : PL.bd);
    e.c_prev = io.c_prev;
    e.c_out = io.c_out;
    e.h_out = io.h_out;
    e.ldh = HID;
    e.gates_out = io.gates_out;
    e.drop = make_drop(seed, which == 0 ? d.p_att : d.p_dec, training);
    e.site = which == 0 ? SITE_ATT : SITE_DEC;
    e.t = (uint32_t)t;
    e.row_offset = row_offset;
    e.HID = HID;
    return launch_gemm<32, EpiLstm>(g, e, st);
}

int run_query(const Dims &d, const gvx_weights *w, const float *h_att, int B, float *q, cudaStream_t st) {
    GemmIn g = gemm_in(w->query_w, d.A, d.D, B);
    add_seg(g, h_att, d.A, d.A);
    EpiStore e;
    memset(&e, 0, sizeof(e));
    e.out = q;
    e.ldo = d.D;
    return launch_gemm<8, EpiStore>(g, e, st);
}

int run_attention(const Dims &d, const gvx_weights *w, const float *packed, const float *q, const float *pm,
                  const float *memory, const int64_t *lengths, int B, int N, float *w_prev, float *cum, float *align_out,
                  long long align_bstride, float *cum_stash, float *ctx_out, float *th_stash, float *conv_stash,
                  cudaStream_t st) {
    const PackedL PL(d);
    AttnFwdArgs a;
    memset(&a, 0, sizeof(a));
    a.s = AttnShape{B, N, d.D, d.E, d.F, d.KS};
    a.q = src_plain(q, d.D); a.pm = pm; a.memory = memory;
    a.wlc = w->loc_conv_w; a.wldT = packed + PL.wldT; a.v = w->v_w;
    a.lengths = lengths;
    a.w_prev = w_prev; a.cum = cum;
    a.align_out = align_out; a.align_bstride = align_bstride; a.cum_stash = cum_stash;
    a.ctx_out = ctx_out; a.ctx_ld = d.E;
    a.th_stash = th_stash; a.conv_stash = conv_stash;
    return launch_attention_fwd_best(a, st);
}

// [mel | gate] = [h_dec, ctx] . Wpg^T + bpg   (tacotron2.py:360-362) over `rows` rows
int run_projection(const Dims &d, const float *packed, const float *hd, int hd_ld, const float *ctx, int ctx_ld, int rows,
                   float *out, cudaStream_t st, bool small) {
    const PackedL PL(d);
    GemmIn g = gemm_in(packed + PL.Wpg, d.Kp, d.M + 1, rows);
    add_seg(g, hd, d.H, hd_ld);
    add_seg(g, ctx, d.E, ctx_ld);
    EpiStore e;
    memset(&e, 0, sizeof(e));
    e.out = out;
    e.ldo = d.OL;
    e.bias = packed + PL.bpg;
    return small ? launch_gemm<8, EpiStore>(g, e, st) : launch_gemm<32, EpiStore>(g, e, st);
}

}  // namespace gvx

using namespace gvx;

extern "C" {

// fingerprint of the sources this library was compiled from (genvox_b200/build.py looks the marker up in the file)
#ifndef GVX_BUILD_FINGERPRINT
#define GVX_BUILD_FINGERPRINT "unknown"
#endif
extern "C" __attribute__((used, visibility("default"))) const char gvx_build_marker[] = "GVXFP:" GVX_BUILD_FINGERPRINT;

int gvx_abi_version(void) { return GVX_ABI_VERSION; }
const char *gvx_last_error(void) { return g_err; }

int gvx_device_info(int *sm_count, int *cc_major, int *cc_minor) {
    int dev = 0;
    GVX_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    GVX_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return 0;
}

unsigned long long gvx_launch_count(void) { return g_launches; }
int gvx_profile_enable(int on) {
    g_prof.on = on ? 1 : 0;
    return 0;
}
int gvx_profile_reset(void) {
    g_prof.collect();
    for (int i = 0; i < PS_NSLOT; ++i) { g_prof.total_ms[i] = 0; g_prof.count[i] = 0; }
    return 0;
}
int gvx_profile_read(int slot, double *total_ms, long long *launches) {
    GVX_CHECK(slot >= 0 && slot < PS_NSLOT, "bad profile slot");
    g_prof.collect();
    if (total_ms) *total_ms = g_prof.total_ms[slot];
    if (launches) *launches = g_prof.count[slot];
    return 0;
}
const char *gvx_profile_slot_name(int slot) { return prof_slot_name(slot); }

size_t gvx_dec_packed_bytes(const gvx_dims *d) {
    if (check_dims(d)) return 0;
    if (d->precision == GVX_BF16) return packed_total_bf16(Dims(*d)) * sizeof(float);
    return PackedL(Dims(*d)).total * sizeof(float);
}

int gvx_dec_pack_weights(const gvx_dims *dd, const gvx_weights *w, void *packed_, void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_, "null argument");
    const Dims d(*dd);
    const PackedL PL(d);
    float *p = (float *)packed_;
    cudaStream_t st = (cudaStream_t)stream;
    k_pack_lstm<<<grid_for((size_t)4 * d.A * d.Ka), 256, 0, st>>>(w->att_w_ih, w->att_w_hh, w->att_b_ih, w->att_b_hh, d.A,
                                                                 d.P + d.E, p + PL.Wa, p + PL.ba, p + PL.WaT);
    GVX_LAUNCHED(1);
    k_pack_lstm<<<grid_for((size_t)4 * d.H * d.Kd), 256, 0, st>>>(w->dec_w_ih, w->dec_w_hh, w->dec_b_ih, w->dec_b_hh, d.H,
                                                                 d.A + d.E, p + PL.Wd, p + PL.bd, p + PL.WdT);
    GVX_LAUNCHED(1);
    k_pack_proj<<<grid_for((size_t)(d.M + 1) * d.Kp), 256, 0, st>>>(w->proj_w, w->proj_b, w->gate_w, w->gate_b, d.M, d.Kp,
                                                                   p + PL.Wpg, p + PL.bpg);
    GVX_LAUNCHED(1);
    k_transpose<<<grid_for((size_t)d.D * d.A), 256, 0, st>>>(w->query_w, d.D, d.A, p + PL.WqT);
    GVX_LAUNCHED(1);
    k_transpose<<<grid_for((size_t)d.D * d.F), 256, 0, st>>>(w->loc_dense_w, d.D, d.F, p + PL.wldT);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    if (dd->precision == GVX_BF16) return pack_weights_bf16(d, w, p, st);
    return 0;
}

size_t gvx_dec_stash_bytes(const gvx_dims *d, int B, int N, int T) {
    if (check_dims(d) || B <= 0 || N <= 0 || T <= 0) return 0;
    if (d->precision == GVX_BF16) return stash_total_bf16(Dims(*d), B, N, T) * sizeof(float);
    return StashL(Dims(*d), B, N, T).total * sizeof(float);
}
size_t gvx_dec_bwd_workspace_bytes(const gvx_dims *d, int B, int N, int T) {
    if (check_dims(d) || B <= 0 || N <= 0 || T <= 0) return 0;
    if (d->precision == GVX_BF16) return bwd_total_bf16(Dims(*d), B, N, T) * sizeof(float);
    return BwdL(Dims(*d), B, N, T).total * sizeof(float);
}
size_t gvx_dec_infer_workspace_bytes(const gvx_dims *d, int B, int N, int max_steps) {
    if (check_dims(d) || B <= 0 || N <= 0 || max_steps <= 0) return 0;
    if (d->precision == GVX_BF16) return infer_total_bf16(Dims(*d), B, N, max_steps) * sizeof(float);
    return InferL(Dims(*d), B, N, max_steps).total * sizeof(float);
}

static int train_fwd_body(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                          const float *mel_in, const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training,
                          int row_offset, float *mel_out, float *gate_out, float *align_out, void *stash_, void *stream) {
    const Dims d(*dd);
    if (dd->precision == GVX_BF16)
        return train_fwd_bf16(d, w, (const float *)packed_, memory, mel_in, mem_lengths, B, N, T, seed, training, row_offset, mel_out,
                              gate_out, align_out, (float *)stash_, (cudaStream_t)stream);
    const StashL S(d, B, N, T);
    const float *packed = (const float *)packed_;
    float *s = (float *)stash_;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H, BE = (size_t)B * d.E;

    // go frame + parse_decoder_inputs, prenet over all frames (tacotron2.py:370-373)
    ProfScope *ps_setup = new ProfScope(PS_SETUP, st);
    k_pack_frames<<<grid_for((size_t)T * B * d.M), 256, 0, st>>>(mel_in, B, d.M, T, s + S.FR);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_TRY(run_prenet(d, w, s + S.FR, d.M, T * B, B, seed, 0, row_offset, s + S.PRE1, s + S.PRE2, st));
    // initialize_decoder_states (tacotron2.py:303-315)
    GVX_TRY(run_processed_memory(d, w, memory, B, N, s + S.PM, st));
    GVX_CUDA(cudaMemsetAsync(s + S.HA, 0, BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CA, 0, BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.HD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CTX, 0, BE * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.WPREV, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + S.CUM, 0, (size_t)B * N * sizeof(float), st));
    delete ps_setup;

    pdl_barrier_next();
    for (int t = 0; t < T; ++t) {   // Decoder.decode, tacotron2.py:333-363
        LstmIO a;
        a.x0 = s + S.PRE2 + (size_t)t * B * d.P; a.w0 = d.P; a.ld0 = d.P;
        a.x1 = s + S.CTX + t * BE; a.w1 = d.E; a.ld1 = d.E;
        a.x2 = s + S.HA + t * BA; a.w2 = d.A; a.ld2 = d.A;
        a.c_prev = s + S.CA + t * BA; a.c_out = s + S.CA + (t + 1) * BA; a.h_out = s + S.HA + (t + 1) * BA;
        a.gates_out = s + S.GA + (size_t)t * 4 * BA;
        { ProfScope ps(PS_ATT_LSTM, st); GVX_TRY(run_lstm(d, packed, 0, a, B, seed, t, training, row_offset, st)); }
        float *q = s + S.Q + (size_t)t * B * d.D;
        { ProfScope ps(PS_QUERY, st); GVX_TRY(run_query(d, w, s + S.HA + (t + 1) * BA, B, q, st)); }
        ProfScope *pa = new ProfScope(PS_ATTENTION, st);
        GVX_TRY(run_attention(d, w, packed, q, s + S.PM, memory, mem_lengths, B, N, s + S.WPREV, s + S.CUM,
                              s + S.ALIGN + (size_t)t * N, (long long)T * N, s + S.CUMS + (size_t)t * N,
                              s + S.CTX + (t + 1) * BE, s + S.TH + (size_t)t * B * N * d.D,
                              s + S.CONVS + (size_t)t * B * N * d.F, st));
        delete pa;
        LstmIO c;
        c.x0 = s + S.HA + (t + 1) * BA; c.w0 = d.A; c.ld0 = d.A;
        c.x1 = s + S.CTX + (t + 1) * BE; c.w1 = d.E; c.ld1 = d.E;
        c.x2 = s + S.HD + t * BH; c.w2 = d.H; c.ld2 = d.H;
        c.c_prev = s + S.CD + t * BH; c.c_out = s + S.CD + (t + 1) * BH; c.h_out = s + S.HD + (t + 1) * BH;
        c.gates_out = s + S.GD + (size_t)t * 4 * BH;
        { ProfScope ps(PS_DEC_LSTM, st); GVX_TRY(run_lstm(d, packed, 1, c, B, seed, t, training, row_offset, st)); }
    }
    ProfScope ps_out(PS_OUTPUT, st);
    // projections for all frames at once, then parse_decoder_outputs (tacotron2.py:360-362,:322-331)
    GVX_TRY(run_projection(d, packed, s + S.HD + BH, d.H, s + S.CTX + BE, d.E, T * B, s + S.OUT, st, false));
    k_unpack_out<<<grid_for((size_t)B * (d.M + 1) * T), 256, 0, st>>>(s + S.OUT, B, d.M, d.OL, T, T, mel_out, gate_out);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_CUDA(cudaMemcpyAsync(align_out, s + S.ALIGN, (size_t)B * T * N * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

// One decoder step of inference (tacotron2.py:398-403): prenet on the previous mel frame `prev` (dropout on, :143), attention
// LSTM, attention (weights to align_t, row stride align_bstride), decoder LSTM, [mel | gate] projection to out_t.
// row_frame / row_id: optional per-row prenet dropout frame and row (run_prenet).
static int infer_step(const Dims &d, const gvx_weights *w, const float *packed, const InferL &L, float *s, const float *memory,
                      const int64_t *mem_lengths, int B, int N, uint64_t seed, int t, int training, int row_offset,
                      const int *row_frame, const int *row_id, const float *prev, float *align_t, long long align_bstride,
                      float *out_t, bool fused_prenet, cudaStream_t st) {
    const int cur = t & 1, nxt = cur ^ 1;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H;
    int *flags = (int *)(s + L.FLAGS);
    { ProfScope ps(PS_PRENET, st);
      if (fused_prenet) {
          GVX_TRY(run_infer_prenet(d, w, prev, d.OL, B, seed, t, row_offset, s + L.PRE1, s + L.PRE2, nullptr, (unsigned *)(flags + 40), flags + 41, st,
                                   row_frame, row_id));
      } else {
          GVX_TRY(run_prenet(d, w, prev, d.OL, B, B, seed, t, row_offset, s + L.PRE1, s + L.PRE2, st, nullptr, row_frame, row_id));
      } }
    LstmIO a;
    a.x0 = s + L.PRE2; a.w0 = d.P; a.ld0 = d.P;
    a.x1 = s + L.CTX; a.w1 = d.E; a.ld1 = d.E;
    a.x2 = s + L.HA + cur * BA; a.w2 = d.A; a.ld2 = d.A;
    a.c_prev = s + L.CA; a.c_out = s + L.CA; a.h_out = s + L.HA + nxt * BA; a.gates_out = nullptr;
    { ProfScope ps(PS_ATT_LSTM, st); GVX_TRY(run_lstm(d, packed, 0, a, B, seed, t, training, row_offset, st)); }
    { ProfScope ps(PS_QUERY, st); GVX_TRY(run_query(d, w, s + L.HA + nxt * BA, B, s + L.Q, st)); }
    { ProfScope ps(PS_ATTENTION, st);
      GVX_TRY(run_attention(d, w, packed, s + L.Q, s + L.PM, memory, mem_lengths, B, N, s + L.WPREV, s + L.CUM,
                            align_t, align_bstride, nullptr, s + L.CTX, nullptr, nullptr, st)); }
    LstmIO c;
    c.x0 = s + L.HA + nxt * BA; c.w0 = d.A; c.ld0 = d.A;
    c.x1 = s + L.CTX; c.w1 = d.E; c.ld1 = d.E;
    c.x2 = s + L.HD + cur * BH; c.w2 = d.H; c.ld2 = d.H;
    c.c_prev = s + L.CD; c.c_out = s + L.CD; c.h_out = s + L.HD + nxt * BH; c.gates_out = nullptr;
    { ProfScope ps(PS_DEC_LSTM, st); GVX_TRY(run_lstm(d, packed, 1, c, B, seed, t, training, row_offset, st)); }
    { ProfScope ps(PS_PROJ, st); GVX_TRY(run_projection(d, packed, s + L.HD + nxt * BH, d.H, s + L.CTX, d.E, B, out_t, st, true)); }
    return 0;
}

static int infer_body(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                      const int64_t *mem_lengths, int B, int N, int max_steps, float gate_threshold, int ignore_gate,
                      uint64_t seed, int training, int row_offset, float *mel_out, float *gate_out, float *align_out,
                      int32_t *n_frames, int *steps_run, void *workspace, void *stream) {
    const Dims d(*dd);
    if (dd->precision == GVX_BF16)
        return infer_bf16(d, w, (const float *)packed_, memory, mem_lengths, B, N, max_steps, gate_threshold, ignore_gate, seed,
                          training, row_offset, mel_out, gate_out, align_out, n_frames, steps_run, (float *)workspace,
                          (cudaStream_t)stream);
    const InferL L(d, B, N, max_steps);
    const float *packed = (const float *)packed_;
    float *s = (float *)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H;
    int *flags = (int *)(s + L.FLAGS);

    GVX_TRY(run_processed_memory(d, w, memory, B, N, s + L.PM, st));
    GVX_CUDA(cudaMemsetAsync(s + L.HA, 0, 2 * BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CA, 0, BA * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.HD, 0, 2 * BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CD, 0, BH * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CTX, 0, (size_t)B * d.E * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.WPREV, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.CUM, 0, (size_t)B * N * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + L.ZERO, 0, (size_t)B * d.OL * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(flags, 0, 32 * sizeof(int), st));       // [0] rows still running; [32..33] hold the dropout seed (gvx_dec_infer)
    GVX_CUDA(cudaMemsetAsync(flags + 40, 0, 2 * sizeof(int), st));   // [40] prenet grid barrier, [41] its error word
    k_fill_i32<<<grid_for(B), 256, 0, st>>>(n_frames, B, ignore_gate ? max_steps : -1, 0);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    const bool fused_prenet = infer_prenet_fused_ok(d, B);

    int t = 0, host_running = B;
    pdl_barrier_next();
    for (; t < max_steps; ++t) {
        const float *prev = t == 0 ? s + L.ZERO : s + L.OUT + (size_t)(t - 1) * B * d.OL;
        float *out_t = s + L.OUT + (size_t)t * B * d.OL;
        GVX_TRY(infer_step(d, w, packed, L, s, memory, mem_lengths, B, N, seed, t, training, row_offset, nullptr, nullptr, prev,
                           align_out + (size_t)t * N, (long long)max_steps * N, out_t, fused_prenet, st));
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
    if (!ignore_gate) {   // rows that never fired stop at max_decoder_steps (tacotron2.py:407)
        k_fill_i32<<<grid_for(B), 256, 0, st>>>(n_frames, B, steps, 1);
    GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
    }
    k_unpack_out<<<grid_for((size_t)B * (d.M + 1) * steps), 256, 0, st>>>(s + L.OUT, B, d.M, d.OL, steps, max_steps, mel_out,
                                                                         gate_out);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    *steps_run = steps;
    return 0;
}

// ---------------------------------------------------------------- graph-cached entry points
static uint32_t *seed_slot_train(const gvx_dims *dd, void *stash, int B, int N, int T) {
    const Dims d(*dd);
    const size_t off = dd->precision == GVX_BF16 ? stash_seed_off_bf16(d, B, N, T) : StashL(d, B, N, T).SEED;
    return reinterpret_cast<uint32_t *>((float *)stash + off);
}
static int put_seed(uint32_t *slot, uint64_t seed, cudaStream_t st) {
    k_set_seed<<<1, 1, 0, st>>>(slot, (uint32_t)(seed & 0xffffffffull), (uint32_t)(seed >> 32));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

int gvx_dec_train_fwd(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                      const float *mel_in, const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training,
                      int row_offset, float *mel_out, float *gate_out, float *align_out, void *stash_, void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_ && memory && mel_in && mel_out && gate_out && align_out && stash_, "null argument");
    GVX_CHECK(B > 0 && N > 0 && T > 0, "B, N, T must be positive");
    GVX_TRY(latch_check());
    cudaStream_t user = (cudaStream_t)stream;
    uint32_t *slot = seed_slot_train(dd, stash_, B, N, T);
    GVX_TRY(put_seed(slot, seed, user));
    KeyBuilder kb;
    kb.add((int)1).add(*dd).add(*w).add(packed_).add(memory).add(mel_in).add(mem_lengths).add(B).add(N).add(T).add(training)
        .add(row_offset).add(mel_out).add(gate_out).add(align_out).add(stash_);
    g_seed_ptr = slot;
    const int rc = run_cached(kb.k, user, [&](cudaStream_t st) {
        return train_fwd_body(dd, w, packed_, memory, mel_in, mem_lengths, B, N, T, seed, training, row_offset, mel_out, gate_out,
                              align_out, stash_, (void *)st);
    });
    g_seed_ptr = nullptr;
    return rc;
}

int gvx_dec_infer(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                  const int64_t *mem_lengths, int B, int N, int max_steps, float gate_threshold, int ignore_gate,
                  uint64_t seed, int training, int row_offset, float *mel_out, float *gate_out, float *align_out,
                  int32_t *n_frames, int *steps_run, void *workspace, void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_ && memory && mel_out && gate_out && align_out && n_frames && steps_run && workspace,
              "null argument");
    GVX_CHECK(B > 0 && N > 0 && max_steps > 0, "B, N, max_steps must be positive");
    GVX_TRY(latch_check());
    cudaStream_t user = (cudaStream_t)stream;
    const Dims d(*dd);
    const bool bf = dd->precision == GVX_BF16;
    const size_t flags_off = bf ? infer_flags_off_bf16(d, B, N, max_steps) : InferL(d, B, N, max_steps).FLAGS;
    // the seed slot sits behind the stop flags; the drivers only clear the first 32 ints of that block
    uint32_t *slot = reinterpret_cast<uint32_t *>((float *)workspace + flags_off) + 32;
    GVX_TRY(put_seed(slot, seed, user));
    g_seed_ptr = slot;
    int rc;
    if (ignore_gate) {          // fixed step count: no host polling inside, the whole sequence is one graph
        KeyBuilder kb;
        kb.add((int)3).add(*dd).add(*w).add(packed_).add(memory).add(mem_lengths).add(B).add(N).add(max_steps).add(gate_threshold)
            .add(training).add(row_offset).add(mel_out).add(gate_out).add(align_out).add(n_frames).add(workspace);
        rc = run_cached(kb.k, user, [&](cudaStream_t st) {
            return infer_body(dd, w, packed_, memory, mem_lengths, B, N, max_steps, gate_threshold, ignore_gate, seed, training,
                              row_offset, mel_out, gate_out, align_out, n_frames, steps_run, workspace, (void *)st);
        });
        *steps_run = max_steps;
    } else {
        rc = infer_body(dd, w, packed_, memory, mem_lengths, B, N, max_steps, gate_threshold, ignore_gate, seed, training,
                        row_offset, mel_out, gate_out, align_out, n_frames, steps_run, workspace, stream);
    }
    g_seed_ptr = nullptr;
    if (rc == 0 && bf)
        rc = check_tc_err_public(reinterpret_cast<int *>((float *)workspace + infer_err_off_bf16(d, B, N, max_steps)), user,
                                 "gvx_dec_infer");
    if (rc == 0 && !bf)      // error word of the fused inference prenet's grid barrier (gvx_infer_prenet.cuh)
        rc = check_tc_err_public(reinterpret_cast<int *>((float *)workspace + flags_off) + 41, user, "gvx_dec_infer (prenet barrier)");
    return rc;
}

int gvx_device_error(int clear) {
    if (latch_ready()) return -1;
    const int e = *reinterpret_cast<volatile int *>(err_latch_host());
    if (clear) *reinterpret_cast<volatile int *>(err_latch_host()) = 0;
    return e;
}

int gvx_graph_stats(unsigned long long *out4) {
    GVX_CHECK(out4 != nullptr, "null argument");
    out4[0] = g_graph_stats.eager; out4[1] = g_graph_stats.captured; out4[2] = g_graph_stats.replayed;
    out4[3] = g_graph_stats.capture_failed;
    return 0;
}

// ---------------------------------------------------------------- single-phase hooks
int gvx_test_tc_gemm(const float *W, const float *X, int B, int Mtot, int K, int KS, float *out, void *stream) {
    GVX_CHECK(W && X && out && B > 0 && Mtot > 0 && K > 0 && KS > 0, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int NPAD = tc_npad(B);
    GVX_CHECK(NPAD > 0, "batch too large");
    const int Kpad = (K + TC_KB - 1) / TC_KB * TC_KB, Mtiles = (Mtot + TC_M - 1) / TC_M, ldp = Mtiles * TC_M;
    __nv_bfloat16 *wimg = nullptr, *ximg = nullptr;
    float *P = nullptr;
    int *err = nullptr;
    GVX_CUDA(cudaMalloc(&wimg, (size_t)Mtiles * TC_M * Kpad * 2));
    GVX_CUDA(cudaMalloc(&ximg, (size_t)NPAD * Kpad * 2));
    GVX_CUDA(cudaMalloc(&P, (size_t)KS * B * ldp * 4));
    GVX_CUDA(cudaMalloc(&err, 4));
    GVX_CUDA(cudaMemsetAsync(err, 0, 4, st));
    TcPackW pw;
    memset(&pw, 0, sizeof(pw));
    pw.s0 = W; pw.mode = 0; pw.Mtot = Mtot; pw.K = K; pw.ld = K;
    k_tc_pack_w<<<grid_for((size_t)Mtiles * TC_M * Kpad), 256, 0, st>>>(pw, Mtiles, Kpad, wimg);
    k_tc_pack_x<<<grid_for((size_t)NPAD * Kpad), 256, 0, st>>>(X, B, K, K, NPAD, Kpad, ximg);
    TcGemmArgs a;
    memset(&a, 0, sizeof(a));
    a.Wimg = wimg; a.Ximg = ximg; a.P = P; a.Kpad = Kpad; a.B = B; a.ldp = ldp; a.KS = KS; a.err = err;
    int rc = launch_tc_gemm(a, Mtiles, st);
    if (!rc) {
        k_tc_sum_partials<<<grid_for((size_t)B * Mtot), 256, 0, st>>>(P, KS, B, ldp, Mtot, out, Mtot);
        int herr = 0;
        cudaError_t e = cudaMemcpyAsync(&herr, err, 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "tc gemm test: %s", cudaGetErrorString(e)); rc = 1; }
        else if (herr) { snprintf(g_err, sizeof(g_err), "tc gemm pipeline timeout, code %d", herr); rc = 1; }
    }
    cudaFree(wimg); cudaFree(ximg); cudaFree(P); cudaFree(err);
    return rc;
}

int gvx_prenet_fwd(const gvx_dims *dd, const gvx_weights *w, const float *frames, int F, int B, uint64_t seed, int t0,
                   int row_offset, float *tmp, float *out, void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && frames && tmp && out && F > 0 && B > 0, "bad argument");
    const Dims d(*dd);
    return run_prenet(d, w, frames, d.M, F * B, B, seed, t0, row_offset, tmp, out, (cudaStream_t)stream);
}

int gvx_lstm_step(const gvx_dims *dd, const void *packed, int which, const float *x, const float *h, const float *c, int B,
                  uint64_t seed, int t, int training, int row_offset, float *h_out, float *c_out, float *gates_out,
                  void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(packed && x && h && c && h_out && c_out && B > 0 && (which == 0 || which == 1), "bad argument");
    const Dims d(*dd);
    const int HID = which == 0 ? d.A : d.H, K = which == 0 ? d.Ka : d.Kd, IN = K - HID;
    LstmIO io;
    io.x0 = x; io.w0 = IN; io.ld0 = IN;
    io.x1 = h; io.w1 = HID; io.ld1 = HID;
    io.x2 = nullptr; io.w2 = 0; io.ld2 = 0;
    io.c_prev = c; io.c_out = c_out; io.h_out = h_out; io.gates_out = gates_out;
    return run_lstm(d, (const float *)packed, which, io, B, seed, t, training, row_offset, (cudaStream_t)stream);
}

int gvx_attention_step(const gvx_dims *dd, const gvx_weights *w, const void *packed, const float *h_att,
                       const float *memory, const float *processed_memory, const int64_t *mem_lengths, int B, int N,
                       float *w_prev, float *w_cum, float *q_tmp, float *ctx_out, float *align_out, void *stream) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed && h_att && memory && processed_memory && w_prev && w_cum && q_tmp && ctx_out && align_out &&
                  B > 0 && N > 0,
              "bad argument");
    const Dims d(*dd);
    cudaStream_t st = (cudaStream_t)stream;
    GVX_TRY(run_query(d, w, h_att, B, q_tmp, st));
    return run_attention(d, w, (const float *)packed, q_tmp, processed_memory, memory, mem_lengths, B, N, w_prev, w_cum,
                         align_out, (long long)N, nullptr, ctx_out, nullptr, nullptr, st);
}

}  // extern "C"

// backward through time (gvx_dec_train_bwd) lives in its own file, same translation unit
#include "gvx_bwd.cuh"
#include "gvx_bf16_api.cuh"
#include "gvx_continuous.cuh"
#include "gvx_session.cuh"
