// genvox_b200 — decoder sessions: continuous batching for utterances submitted over time, frames returned per step call.
//
// A session is gvx_dec_infer_continuous cut into calls.  Its slots, their recurrent state and a ring of queued utterances
// live in the caller's workspace, and the host struct (gvx_session) holds the counters.  Submit appends to the ring and
// computes processed memory; a step call first admits queued utterances into the idle slots (k_gate_admit in head mode),
// then runs the continuous loop's launch sequence (full dependency, step, k_gate_admit) for up to k steps, writing every
// slot's row of every step into the caller's chunk buffers.
//
// State that survives between calls, all in the workspace: the two-frame output ring (the previous frame of the next step),
// the utt / frame / next / frame-cap ping-pong (current half: gvx_session.parity), the fp32 h / c / ctx / attention rows or, in bf16,
// the cell states and operand images (current half: the parity of steps_run), the seed words (written once at init) and
// the error words.  Two words need care:
//   - the fused prenet's grid barrier (flags[40]) is a monotonic counter that launch t waits on to reach 32 (t + 1); the
//     head admission rewinds it, so that over a long session it never wraps;
//   - the int t of the step functions: with per-row frame and row arrays and no LSTM-state dropout (eval mode), only its
//     parity (the ping-pong halves) and the barrier target use it, so a call passes t = (steps_run & 1) + i.
#pragma once
#include "gvx_continuous.cuh"

namespace gvx {

constexpr int32_t SESSION_READY = 0x53455353;

// workspace: the static inference layout for S rows and a two-frame output ring, then this block
struct SessL {
    size_t MEM, STG, STGP, RMEM, RPM, RLEN, RCAP, ALIGN, LEN, ST, CTL, total;
    SessL(const Dims &d, size_t base, int N, int S, int cap) {
        Carver c;
        c.o = base;
        MEM = c.take((size_t)S * N * d.E);       // [S][N][E] encoder memory of the utterance in each slot
        STG = c.take((size_t)S * N * d.E);       // [S][N][E] one submitted group, zero-padded to S rows
        STGP = c.take((size_t)S * N * d.D);      // [S][N][D] its processed memory
        RMEM = c.take((size_t)cap * N * d.E);    // ring: [cap][N][E] memory, [cap][N][D] processed memory,
        RPM = c.take((size_t)cap * N * d.D);     //       [cap] int64 length, [cap] int32 frame cap; id at id % cap
        RLEN = c.take((size_t)2 * cap);
        RCAP = c.take((size_t)cap);
        ALIGN = c.take((size_t)S * N);           // [S][N] attention weights of the current step
        LEN = c.take((size_t)2 * S);             // [S] int64 memory length of each slot
        ST = c.take((size_t)6 * S + 2);          // int: utt[2][S], frame[2][S], next[2], frame cap[2][S]
        CTL = c.take(4);                         // int: active slots, admission head, finished utterances
        total = c.o;
    }
};

inline SessL session_layout(const Dims &d, bool bf, int N, int S, int cap) {
    return SessL(d, continuous_base(d, bf, S, N), N, S, cap);
}

// length and frame cap of ids first .. first + k - 1 into the ring
__global__ void k_session_put(int64_t *__restrict__ rlen, int32_t *__restrict__ rcap, const int64_t *__restrict__ lengths,
                              const int32_t *__restrict__ caps, int k, long long first, int cap, int N, int max_steps) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < k; i += gridDim.x * blockDim.x) {
        const size_t e = (size_t)((first + i) % cap);
        rlen[e] = lengths ? lengths[i] : (int64_t)N;
        rcap[e] = caps ? caps[i] : max_steps;
    }
}

inline int check_session(const gvx_dims *dd, const gvx_session *s) {
    GVX_TRY(check_dims(dd));
    GVX_CHECK(s != nullptr, "session is null");
    GVX_CHECK(s->N > 0 && s->slots > 0 && s->capacity > 0 && s->max_steps > 0, "session: N, slots, capacity, max_steps must be positive");
    GVX_CHECK(s->row_offset >= 0, "session: row_offset must be non-negative");
    if (dd->precision == GVX_BF16) GVX_TRY(check_bf16_dims(Dims(*dd), s->slots));
    return 0;
}

inline uint32_t *session_seed_slot(const Dims &d, bool bf, int N, int S, float *s) {
    const size_t flags_off = bf ? InferBfL(d, S, N, 2).FLAGS : InferL(d, S, N, 2).FLAGS;
    return reinterpret_cast<uint32_t *>(s + flags_off) + 32;
}

int session_submit(const Dims &d, bool bf, const gvx_weights *w, const gvx_session *ss, const float *memory,
                   const int64_t *lengths, const int32_t *caps, int k, float *s, cudaStream_t st) {
    const int S = ss->slots, N = ss->N, cap = ss->capacity;
    const SessL L = session_layout(d, bf, N, S, cap);
    const size_t NE = (size_t)N * d.E, ND = (size_t)N * d.D;
    // processed memory in launches of exactly S x N rows (the static call's row count, so every row gets the bits the
    // static call computes), through staging buffers: the slot-memory buffer holds live state
    for (int g0 = 0; g0 < k; g0 += S) {
        const int n = k - g0 < S ? k - g0 : S;
        const float *src = memory + (size_t)g0 * NE;
        if (n < S) {
            GVX_CUDA(cudaMemsetAsync(s + L.STG, 0, S * NE * sizeof(float), st));
            GVX_CUDA(cudaMemcpyAsync(s + L.STG, src, n * NE * sizeof(float), cudaMemcpyDeviceToDevice, st));
            src = s + L.STG;
        }
        GVX_TRY(run_processed_memory(d, w, src, S, N, s + L.STGP, st));
        // into the ring: at most two pieces, the second one wrapping to entry 0
        const long long id0 = ss->submitted + g0;
        for (int done = 0; done < n;) {
            const int e = (int)((id0 + done) % cap), m = n - done < cap - e ? n - done : cap - e;
            GVX_CUDA(cudaMemcpyAsync(s + L.RMEM + e * NE, memory + (size_t)(g0 + done) * NE, m * NE * sizeof(float),
                                     cudaMemcpyDeviceToDevice, st));
            GVX_CUDA(cudaMemcpyAsync(s + L.RPM + e * ND, s + L.STGP + done * ND, m * ND * sizeof(float), cudaMemcpyDeviceToDevice, st));
            done += m;
        }
    }
    k_session_put<<<grid_for(k), 256, 0, st>>>((int64_t *)(s + L.RLEN), (int32_t *)(s + L.RCAP), lengths, caps, k, ss->submitted,
                                               cap, N, ss->max_steps);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    return 0;
}

int session_step(const Dims &d, bool bf, const gvx_weights *w, const float *packed, gvx_session *ss, int K, float *frames,
                 float *align, int32_t *utt_out, int32_t *frame_out, int8_t *last_out, int *steps_run, float *s, cudaStream_t st) {
    const int S = ss->slots, N = ss->N, cap = ss->capacity;
    const InferL Lf(d, S, N, 2);
    const InferBfL Lb(d, S, N, 2);
    const SessL L = session_layout(d, bf, N, S, cap);
    const size_t PM = bf ? Lb.PM : Lf.PM, OUT = bf ? Lb.OUT : Lf.OUT, FLAGS = bf ? Lb.FLAGS : Lf.FLAGS;
    int *state = (int *)(s + L.ST), *ctl = (int *)(s + L.CTL);
    int64_t *len_slot = (int64_t *)(s + L.LEN);
    float *mem_slot = s + L.MEM;
    const bool fused_prenet = infer_prenet_fused_ok(d, S);

    AdmitArgs a;
    memset(&a, 0, sizeof(a));
    admit_state(a, d, bf, Lf, Lb, s, S, N);
    a.align_t = s + L.ALIGN;
    a.memory = s + L.RMEM; a.pmq = s + L.RPM; a.lengths = (const int64_t *)(s + L.RLEN); a.caps = (const int32_t *)(s + L.RCAP);
    a.mem_slot = mem_slot; a.pm_slot = s + PM; a.len_slot = len_slot;
    a.ch_frames = frames; a.ch_align = ss->with_alignments ? align : nullptr;
    a.ch_utt = utt_out; a.ch_frame = frame_out; a.ch_last = last_out;
    a.flags = ctl;
    a.thr = ss->gate_threshold;
    a.ignore_gate = ss->ignore_gate; a.S = S; a.N = N; a.E = d.E; a.D = d.D; a.M = d.M; a.OL = d.OL; a.max_steps = ss->max_steps;
    a.U = (int)ss->submitted; a.cap = cap;

    const int hp = (int)(ss->steps_run & 1);       // parity of the h / c ping-pong and of the output ring
    int up = ss->parity;                           // current half of the utt / frame / next / cap ping-pong
    auto slots_at = [&](int half) {
        a.utt_cur = state + half * S; a.frame_cur = state + 2 * S + half * S; a.next_cur = state + 4 * S + half;
        a.utt_nxt = state + (half ^ 1) * S; a.frame_nxt = state + 2 * S + (half ^ 1) * S; a.next_nxt = state + 4 * S + (half ^ 1);
        a.cap_cur = state + 4 * S + 2 + half * S; a.cap_nxt = state + 4 * S + 2 + (half ^ 1) * S;
    };
    // head of the call: the idle slots take queued utterances in slot order; their go frames are zeroed in the ring entry
    // the first step reads.  The queue only grows between calls, so once this admission has run, a slot that goes idle
    // during the call does so because the queue is empty: idle slots and queued utterances never coexist inside a call.
    a.head = 1;
    a.out_t = s + OUT + (size_t)(hp ^ 1) * S * d.OL;
    a.bar = fused_prenet ? (unsigned *)(s + FLAGS) + 40 : nullptr;
    a.bar_value = (unsigned)(d.P / IPN_COLS) * (unsigned)hp;
    slots_at(up);
    pdl_barrier_next();
    GVX_CUDA(launch_pdl(k_gate_admit, dim3(S), dim3(ADMIT_THREADS), 0, st, a));
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    up ^= 1;
    a.head = 0;
    a.bar = nullptr;

    int host[3] = {ss->active, (int)ss->admitted, (int)ss->finished};
    int i = 0;
    for (; i < K; ++i) {
        const int t = hp + i, p = t & 1;
        const float *prev = s + OUT + (size_t)(p ^ 1) * S * d.OL;
        float *out_t = s + OUT + (size_t)p * S * d.OL;
        slots_at(up);
        // full dependency on the previous k_gate_admit, as in the continuous loop (an admission rewrites lengths and
        // processed memory that kernels of the chain read before griddepcontrol.wait)
        pdl_barrier_next();
        if (bf) GVX_TRY(infer_step_bf16(d, w, packed, Lb, s, mem_slot, len_slot, S, N, ss->seed, t, 0, ss->row_offset, a.frame_cur,
                                        a.utt_cur, prev, s + L.ALIGN, (long long)N, out_t, st));
        else GVX_TRY(infer_step(d, w, packed, Lf, s, mem_slot, len_slot, S, N, ss->seed, t, 0, ss->row_offset, a.frame_cur, a.utt_cur,
                                prev, s + L.ALIGN, (long long)N, out_t, fused_prenet, st));
        a.out_t = out_t;
        a.step = i;
        GVX_CUDA(launch_pdl(k_gate_admit, dim3(S), dim3(ADMIT_THREADS), 0, st, a));
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
        up ^= 1;
        if ((i + 1) % GVX_STOP_POLL == 0 || i + 1 == K) {
            GVX_CUDA(cudaMemcpyAsync(host, ctl, sizeof(host), cudaMemcpyDeviceToHost, st));
            GVX_CUDA(cudaStreamSynchronize(st));
            if (host[0] == 0) { ++i; break; }
        }
    }
    *steps_run = i;
    ss->steps_run += i;
    ss->parity = up;
    ss->active = host[0];
    ss->admitted = host[1];
    ss->finished = host[2];
    return 0;
}

}  // namespace gvx

extern "C" {

size_t gvx_dec_session_workspace_bytes(const gvx_dims *d, int N, int slots, int capacity) {
    using namespace gvx;
    if (check_dims(d) || N <= 0 || slots <= 0 || capacity <= 0) return 0;
    const Dims dm(*d);
    const bool bf = d->precision == GVX_BF16;
    if (bf && check_bf16_dims(dm, slots)) return 0;
    return session_layout(dm, bf, N, slots, capacity).total * sizeof(float);
}

int gvx_dec_session_init(const gvx_dims *dd, gvx_session *ss, void *workspace, void *stream) {
    using namespace gvx;
    GVX_TRY(check_session(dd, ss));
    GVX_CHECK(workspace != nullptr, "null argument");
    GVX_TRY(latch_check());
    const Dims d(*dd);
    const bool bf = dd->precision == GVX_BF16;
    const int S = ss->slots, N = ss->N;
    const SessL L = session_layout(d, bf, N, S, ss->capacity);
    float *s = (float *)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    GVX_CUDA(cudaMemsetAsync(s, 0, L.total * sizeof(float), st));      // every slot's state, the output ring, the error words
    k_slot_start<<<grid_for(S), 256, 0, st>>>(S, 0, N, nullptr, (int64_t *)(s + L.LEN), (int *)(s + L.ST));   // all idle
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());
    GVX_TRY(put_seed(session_seed_slot(d, bf, N, S, s), ss->seed, st));
    ss->steps_run = ss->submitted = ss->admitted = ss->finished = 0;
    ss->active = 0;
    ss->parity = 0;
    ss->ready = SESSION_READY;
    return 0;
}

int gvx_dec_session_submit(const gvx_dims *dd, const gvx_weights *w, const void *packed, gvx_session *ss, const float *memory,
                           const int64_t *lengths, const int32_t *frame_caps, int k, void *workspace, void *stream) {
    using namespace gvx;
    GVX_TRY(check_session(dd, ss));
    GVX_CHECK(ss->ready == SESSION_READY, "session: gvx_dec_session_init has not run");
    GVX_CHECK(w && packed && memory && workspace, "null argument");
    GVX_CHECK(k > 0, "session: k must be positive");
    GVX_CHECK(ss->submitted + k - ss->admitted <= ss->capacity, "session: the queue ring is full (submitted + k - admitted > capacity)");
    GVX_CHECK(ss->submitted + k - 1 + ss->row_offset <= 2147483647LL, "session: utterance id + row_offset would pass 2^31 - 1");
    GVX_TRY(latch_check());
    GVX_TRY(session_submit(Dims(*dd), dd->precision == GVX_BF16, w, ss, memory, lengths, frame_caps, k, (float *)workspace,
                           (cudaStream_t)stream));
    ss->submitted += k;
    return 0;
}

int gvx_dec_session_step(const gvx_dims *dd, const gvx_weights *w, const void *packed, gvx_session *ss, int max_steps_this_call,
                         float *frames, float *align, int32_t *utt, int32_t *frame, int8_t *last, int *steps_run, void *workspace,
                         void *stream) {
    using namespace gvx;
    GVX_TRY(check_session(dd, ss));
    GVX_CHECK(ss->ready == SESSION_READY, "session: gvx_dec_session_init has not run");
    GVX_CHECK(w && packed && frames && utt && frame && last && steps_run && workspace, "null argument");
    GVX_CHECK(align || !ss->with_alignments, "session: align is null but with_alignments is set");
    GVX_CHECK(max_steps_this_call > 0, "session: max_steps_this_call must be positive");
    *steps_run = 0;
    if (ss->active == 0 && ss->submitted == ss->admitted) return 0;      // nothing queued, nothing running
    GVX_TRY(latch_check());
    const Dims d(*dd);
    const bool bf = dd->precision == GVX_BF16;
    cudaStream_t st = (cudaStream_t)stream;
    float *s = (float *)workspace;
    g_seed_ptr = session_seed_slot(d, bf, ss->N, ss->slots, s);
    int rc = session_step(d, bf, w, (const float *)packed, ss, max_steps_this_call, frames, align, utt, frame, last, steps_run, s, st);
    g_seed_ptr = nullptr;
    if (rc == 0 && bf)
        rc = check_tc_err_public(reinterpret_cast<int *>(s + InferBfL(d, ss->slots, ss->N, 2).ERR), st, "gvx_dec_session_step");
    if (rc == 0 && !bf)
        rc = check_tc_err_public(reinterpret_cast<int *>(s + InferL(d, ss->slots, ss->N, 2).FLAGS) + 41, st,
                                 "gvx_dec_session_step (prenet barrier)");
    return rc;
}

}  // extern "C"
