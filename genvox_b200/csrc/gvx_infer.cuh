// genvox_b200 — inference: the per-precision plan of an inference workspace, the static decode loop and its entry points.
// The static loop here, the continuous loop (gvx_continuous.cuh) and sessions (gvx_session.cuh) see the precision only
// through InferPlan: its layout, the recurrent state a decode starts from zero, the step function and the error word.
#pragma once
#include "gvx_bf16_api.cuh"

namespace gvx {

// One decoder step of inference (tacotron2.py:398-403): prenet on the previous mel frame io.prev (dropout on, :143), attention
// LSTM, attention, decoder LSTM, [mel | gate] projection to io.out_t.
static int infer_step(const Dims &d, const gvx_weights *w, const float *packed, const InferL &L, float *s, int B, int N,
                      bool fused_prenet, const InferStepArgs &io, cudaStream_t st) {
    const int t = io.t, cur = t & 1, nxt = cur ^ 1;
    const size_t BA = (size_t)B * d.A, BH = (size_t)B * d.H;
    int *flags = (int *)(s + L.FLAGS);
    { ProfScope ps(PS_PRENET, st);
      if (fused_prenet) {
          GVX_TRY(run_infer_prenet(d, w, io.prev, d.OL, B, io.seed, t, io.row_offset, s + L.PRE1, s + L.PRE2, nullptr, (unsigned *)(flags + 40),
                                   flags + 41, st, io.row_frame, io.row_id));
      } else {
          GVX_TRY(run_prenet(d, w, io.prev, d.OL, B, B, io.seed, t, io.row_offset, s + L.PRE1, s + L.PRE2, st, nullptr, io.row_frame,
                             io.row_id));
      } }
    LstmIO a;
    a.x0 = s + L.PRE2; a.w0 = d.P; a.ld0 = d.P;
    a.x1 = s + L.CTX; a.w1 = d.E; a.ld1 = d.E;
    a.x2 = s + L.HA + cur * BA; a.w2 = d.A; a.ld2 = d.A;
    a.c_prev = s + L.CA; a.c_out = s + L.CA; a.h_out = s + L.HA + nxt * BA; a.gates_out = nullptr;
    { ProfScope ps(PS_ATT_LSTM, st); GVX_TRY(run_lstm(d, packed, 0, a, B, io.seed, t, io.training, io.row_offset, st)); }
    { ProfScope ps(PS_QUERY, st); GVX_TRY(run_query(d, w, s + L.HA + nxt * BA, B, s + L.Q, st)); }
    { ProfScope ps(PS_ATTENTION, st);
      GVX_TRY(run_attention(d, w, packed, s + L.Q, s + L.PM, io.memory, io.lengths, B, N, s + L.WPREV, s + L.CUM, io.align_t,
                            io.align_bstride, nullptr, s + L.CTX, nullptr, nullptr, st, io.win_back, io.win_fwd)); }
    LstmIO c;
    c.x0 = s + L.HA + nxt * BA; c.w0 = d.A; c.ld0 = d.A;
    c.x1 = s + L.CTX; c.w1 = d.E; c.ld1 = d.E;
    c.x2 = s + L.HD + cur * BH; c.w2 = d.H; c.ld2 = d.H;
    c.c_prev = s + L.CD; c.c_out = s + L.CD; c.h_out = s + L.HD + nxt * BH; c.gates_out = nullptr;
    { ProfScope ps(PS_DEC_LSTM, st); GVX_TRY(run_lstm(d, packed, 1, c, B, io.seed, t, io.training, io.row_offset, st)); }
    { ProfScope ps(PS_PROJ, st); GVX_TRY(run_projection(d, packed, s + L.HD + nxt * BH, d.H, s + L.CTX, d.E, B, io.out_t, st, true)); }
    return 0;
}

// An inference workspace of B rows, N memory frames and `steps` output frames, in the layout of its precision: InferL in
// fp32, InferBfL in bf16.
struct InferPlan {
    Dims d;
    bool bf;
    int B, N;
    InferL Lf;
    InferBfL Lb;
    size_t PM, OUT, ZERO, FLAGS, total;
    bool fused_prenet;                 // the fused inference prenet runs (infer_prenet_fused_ok)

    InferPlan(const gvx_dims &dd, int rows, int n, int steps)
        : d(dd), bf(dd.precision == GVX_BF16), B(rows), N(n), Lf(d, B, N, steps), Lb(d, B, N, steps),
          PM(bf ? Lb.PM : Lf.PM), OUT(bf ? Lb.OUT : Lf.OUT), ZERO(bf ? Lb.ZERO : Lf.ZERO), FLAGS(bf ? Lb.FLAGS : Lf.FLAGS),
          total(bf ? Lb.total : Lf.total), fused_prenet(infer_prenet_fused_ok(d, B)) {}

    // [0] rows (slots) still running; [32..33] the dropout seed; [40] the fused prenet's grid barrier, [41] its error word
    int *flags(float *s) const { return (int *)(s + FLAGS); }
    uint32_t *seed_slot(float *s) const { return reinterpret_cast<uint32_t *>(flags(s) + 32); }

    // The recurrent state a decode starts from zero, in the layout it lives in: zrow(p, w) for fp32 rows of width w (row r at
    // p + r * w), img(p, kpad) for a tcgen05 operand image ([kpad/64 slabs][Lb.NPAD rows][64], gvx_io.cuh).  fp32: h (both
    // ping-pong halves) and c of both LSTMs, ctx, attention weights and cumulative weights; bf16: the cell states, attention
    // weights and cumulative weights, and the operand images that carry h and ctx.  reset() zeroes all rows of it,
    // k_gate_admit the rows of a slot that takes a new utterance: the two must agree for the continuous and session
    // decodes to be bit-identical to the static one.
    template <class Z, class I> void state(float *s, Z &&zrow, I &&img) const {
        if (bf) {
            const BfGeom g(d);
            zrow(s + Lb.CA, d.A); zrow(s + Lb.CD, d.H); zrow(s + Lb.WPREV, N); zrow(s + Lb.CUM, N);
            bf16 *XAI = (bf16 *)(s + Lb.XAI), *XDI = (bf16 *)(s + Lb.XDI);
            img(XAI, g.Kpa); img(XAI + Lb.xai_stride, g.Kpa);
            img(XDI, g.Kpd); img(XDI + Lb.xdi_stride, g.Kpd);
            img((bf16 *)(s + Lb.XPI), g.Kpp);
        } else {
            zrow(s + Lf.HA, d.A); zrow(s + Lf.HA + (size_t)B * d.A, d.A); zrow(s + Lf.CA, d.A);
            zrow(s + Lf.HD, d.H); zrow(s + Lf.HD + (size_t)B * d.H, d.H); zrow(s + Lf.CD, d.H);
            zrow(s + Lf.CTX, d.E); zrow(s + Lf.WPREV, N); zrow(s + Lf.CUM, N);
        }
    }

    // the recurrent state, flags[0..31], flags[40..41] and the bf16 error words; never the seed words, which put_seed
    // writes before the call's launch sequence
    int reset(float *s, cudaStream_t st) const {
        cudaError_t memset_err = cudaSuccess;
        auto zero = [&](void *p, size_t bytes) { if (memset_err == cudaSuccess) memset_err = cudaMemsetAsync(p, 0, bytes, st); };
        state(s, [&](float *p, int w) { zero(p, (size_t)B * w * sizeof(float)); },
              [&](bf16 *p, int kpad) { zero(p, (size_t)kpad * Lb.NPAD * sizeof(bf16)); });
        zero(flags(s), 32 * sizeof(int));
        zero(flags(s) + 40, 2 * sizeof(int));
        if (bf) zero(s + Lb.ERR, 64 * sizeof(float));
        GVX_CUDA(memset_err);
        return 0;
    }

    int step(const gvx_weights *w, const float *packed, float *s, const InferStepArgs &io, cudaStream_t st) const {
        if (bf) return infer_step_bf16(d, w, packed, Lb, s, B, N, fused_prenet, io, st);
        return infer_step(d, w, packed, Lf, s, B, N, fused_prenet, io, st);
    }

    // after the call: the tcgen05 pipelines' error word in bf16, the fused prenet barrier's in fp32
    int check_err(float *s, cudaStream_t st, const char *what) const {
        if (bf) return check_tc_err((int *)(s + Lb.ERR), st, what);
        char msg[128];
        snprintf(msg, sizeof(msg), "%s (prenet barrier)", what);
        return check_tc_err(flags(s) + 41, st, msg);
    }
};

// The frame of every inference entry point: the dropout seed into the plan's seed slot (a session writes it once, at init),
// the body enqueued with g_seed_ptr at that slot (the dropout of its kernels reads the seed there, so a captured graph
// outlives it), then the plan's error word.
template <class Body>
int infer_call(const InferPlan &P, float *s, bool write_seed, uint64_t seed, cudaStream_t st, const char *what, Body &&body) {
    uint32_t *slot = P.seed_slot(s);
    if (write_seed) GVX_TRY(put_seed(slot, seed, st));
    g_seed_ptr = slot;
    const int rc = body();
    g_seed_ptr = nullptr;
    return rc ? rc : P.check_err(s, st, what);
}

// Decoder.inference (tacotron2.py:390-414) of P.B rows: until every row's gate fired (k_gate_check, polled every GVX_STOP_POLL
// steps) or for max_steps steps (ignore_gate).
static int infer_static(const InferPlan &P, const gvx_weights *w, const float *packed, const float *memory,
                        const int64_t *mem_lengths, int max_steps, float gate_threshold, int ignore_gate, uint64_t seed,
                        int training, int row_offset, float *mel_out, float *gate_out, float *align_out, int32_t *n_frames,
                        int *steps_run, int win_back, int win_fwd, float *s, cudaStream_t st) {
    const Dims &d = P.d;
    const int B = P.B, N = P.N;
    int *flags = P.flags(s);

    GVX_TRY(run_processed_memory(d, w, memory, B, N, s + P.PM, st));
    GVX_TRY(P.reset(s, st));
    GVX_CUDA(cudaMemsetAsync(s + P.ZERO, 0, (size_t)B * d.OL * sizeof(float), st));
    k_fill_i32<<<grid_for(B), 256, 0, st>>>(n_frames, B, ignore_gate ? max_steps : -1, 0);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());

    InferStepArgs io;
    memset(&io, 0, sizeof(io));
    io.memory = memory; io.lengths = mem_lengths;
    io.align_bstride = (long long)max_steps * N;
    io.seed = seed; io.training = training; io.row_offset = row_offset;
    io.win_back = win_back; io.win_fwd = win_fwd;
    int t = 0, host_running = B;
    pdl_barrier_next();
    for (; t < max_steps; ++t) {
        io.t = t;
        io.prev = t == 0 ? s + P.ZERO : s + P.OUT + (size_t)(t - 1) * B * d.OL;
        io.out_t = s + P.OUT + (size_t)t * B * d.OL;
        io.align_t = align_out + (size_t)t * N;
        GVX_TRY(P.step(w, packed, s, io, st));
        if (!ignore_gate) {
            GVX_CUDA(launch_pdl(k_gate_check, dim3(1), dim3(128), 0, st, (const float *)io.out_t, B, d.M, d.OL, gate_threshold, t,
                                n_frames, flags));
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
    k_unpack_out<<<grid_for((size_t)B * (d.M + 1) * steps), 256, 0, st>>>(s + P.OUT, B, d.M, d.OL, steps, max_steps, mel_out,
                                                                         gate_out);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    *steps_run = steps;
    return 0;
}

}  // namespace gvx

extern "C" {

size_t gvx_dec_infer_workspace_bytes(const gvx_dims *d, int B, int N, int max_steps) {
    using namespace gvx;
    if (check_dims(d) || B <= 0 || N <= 0 || max_steps <= 0) return 0;
    return InferPlan(*d, B, N, max_steps).total * sizeof(float);
}

int gvx_dec_infer_windowed(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                           const int64_t *mem_lengths, int B, int N, int max_steps, float gate_threshold, int ignore_gate,
                           uint64_t seed, int training, int row_offset, float *mel_out, float *gate_out, float *align_out,
                           int32_t *n_frames, int *steps_run, int att_backward, int att_forward, void *workspace, void *stream) {
    using namespace gvx;
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_ && memory && mel_out && gate_out && align_out && n_frames && steps_run && workspace,
              "null argument");
    GVX_CHECK(B > 0 && N > 0 && max_steps > 0, "B, N, max_steps must be positive");
    GVX_TRY(check_window(att_backward, att_forward));
    GVX_TRY(latch_check());
    const InferPlan P(*dd, B, N, max_steps);
    if (P.bf) GVX_TRY(check_bf16_dims(P.d, B));
    cudaStream_t user = (cudaStream_t)stream;
    float *s = (float *)workspace;
    auto body = [&](cudaStream_t st) {
        return infer_static(P, w, (const float *)packed_, memory, mem_lengths, max_steps, gate_threshold, ignore_gate, seed, training,
                            row_offset, mel_out, gate_out, align_out, n_frames, steps_run, att_backward, att_forward, s, st);
    };
    return infer_call(P, s, true, seed, user, "gvx_dec_infer", [&] {
        if (!ignore_gate) return body(user);
        // fixed step count: no host polling inside, the whole sequence is one graph
        KeyBuilder kb;
        kb.add((int)3).add(*dd).add(*w).add(packed_).add(memory).add(mem_lengths).add(B).add(N).add(max_steps).add(gate_threshold)
            .add(training).add(row_offset).add(mel_out).add(gate_out).add(align_out).add(n_frames).add(workspace)
            .add(att_backward).add(att_forward);       // baked into the captured attention launches
        const int rc = run_cached(kb.k, user, body);
        *steps_run = max_steps;
        return rc;
    });
}

int gvx_dec_infer(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                  const int64_t *mem_lengths, int B, int N, int max_steps, float gate_threshold, int ignore_gate,
                  uint64_t seed, int training, int row_offset, float *mel_out, float *gate_out, float *align_out,
                  int32_t *n_frames, int *steps_run, void *workspace, void *stream) {
    return gvx_dec_infer_windowed(dd, w, packed_, memory, mem_lengths, B, N, max_steps, gate_threshold, ignore_gate, seed, training,
                                  row_offset, mel_out, gate_out, align_out, n_frames, steps_run, 0, 0, workspace, stream);
}

}  // extern "C"
