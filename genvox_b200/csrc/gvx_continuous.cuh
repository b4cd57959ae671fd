// genvox_b200 — continuous-batching inference: a queue of U utterances decoded through S fixed decoder slots.
//
// Static batching (gvx_dec_infer) runs every batch until its last row stops, so rows that stop early sit idle.  Here a slot
// whose utterance stops takes the next utterance of the queue on the device, before the next decoder step: k_gate_admit runs
// in the launch slot k_gate_check has in the static loop.  Per step it writes each slot's frame straight into its
// utterance's outputs, applies the stop test, admits and resets, and publishes the number of active slots for the host
// poll.  Admission is deterministic and uses no atomics: the slots that stop in the same step take queue entries in slot
// order, and every CTA recomputes all S stop decisions to find its own prefix count.
//
// Output identity: utterance u decodes bit-identically to row r of a static call with the same S rows, N, seed, precision
// and attention window, u in row r and dropout_row_offset = u + row_offset - r.  The slot's every piece of recurrent state is zeroed
// in the layout it lives in, its memory / processed memory / length are replaced, and the prenet draws its dropout at
// Philox (row u + row_offset, t = local frame) through the per-row row_frame / row_id arrays.
#pragma once
#include "gvx_infer.cuh"

namespace gvx {

// ---- workspace: the inference plan's layout for S rows and a two-frame output ring (steps = 2), then this block
struct ContL {
    size_t MEM, PMQ, ALIGN, LEN, ST, total;
    ContL(const Dims &d, size_t base, int U, int N, int S) {
        Carver c;
        c.o = base;
        const size_t Upad = (size_t)(U + S - 1) / S * S;
        MEM = c.take((size_t)S * N * d.E);       // [S][N][E] encoder memory of the utterance in each slot
        PMQ = c.take(Upad * N * d.D);            // [Upad][N][D] processed memory of the whole queue
        ALIGN = c.take((size_t)S * N);           // [S][N] attention weights of the current step
        LEN = c.take((size_t)2 * S);             // [S] int64 memory length of each slot
        ST = c.take((size_t)4 * S + 2);          // int: utt[2][S], frame[2][S], next[2] (ping-pong by step parity)
        total = c.o;
    }
};

constexpr int ADMIT_THREADS = 256;
constexpr int ADMIT_MAXZ = 12;
constexpr int ADMIT_MAXI = 5;

struct AdmitArgs {
    float *out_t;                      // [S][OL] this step's [mel | gate] rows: the previous frame of the next step
    const float *align_t;              // [S][N] this step's attention weights
    const float *memory, *pmq;         // queue entry q at q (cap = 0) or q % cap: [..][N][E], [..][N][D]
    const int64_t *lengths;            // per queue entry, or null (all N)
    const int32_t *caps;               // per queue entry, or null
    float *mem_slot, *pm_slot;         // [S][N][E], [S][N][D]
    int64_t *len_slot;                 // [S]
    const int *utt_cur, *frame_cur, *next_cur;
    int *utt_nxt, *frame_nxt, *next_nxt;
    // session: each slot's frame cap, copied in at admission (a ring entry can be reused while its utterance still runs)
    const int *cap_cur;
    int *cap_nxt;
    float *mel_out, *gate_out, *align_out;   // per-utterance outputs [U][..][max_steps] (continuous call)
    int32_t *n_frames;
    // per-call chunk outputs of a session, used instead of the per-utterance ones when ch_utt is set: row [step][slot]
    float *ch_frames, *ch_align;       // [steps][S][M+1], [steps][S][N] or null
    int32_t *ch_utt, *ch_frame;        // [steps][S] utterance (-1: idle) and its local frame
    int8_t *ch_last;                   // [steps][S] 1 on the utterance's last frame
    int step;
    int *flags;                        // [0] active slots after this step; sessions (cap > 0): [1] admission head, [2] += stops
    unsigned *bar;                     // head mode: the fused prenet's grid-barrier counter, set to bar_value (or null)
    unsigned bar_value;
    float *zero[ADMIT_MAXZ];           // per-row fp32 state, row s at zero[i] + s * zero_w[i]
    int zero_w[ADMIT_MAXZ];
    int nzero;
    __nv_bfloat16 *img[ADMIT_MAXI];    // tcgen05 operand images ([kpad/64 slabs][npad rows][64], gvx_io.cuh)
    int img_k[ADMIT_MAXI];
    int nimg, npad;
    float thr;
    int ignore_gate, S, N, E, D, M, OL, max_steps;
    int U;                             // queue entries q < U exist (a session passes its submitted count)
    int cap;                           // session ring capacity; 0: the queue is a plain array
    int head;                          // 1: admit into idle slots only, before the first step of a session call (no frame)
};

// stop test of gvx_dec_infer (tacotron2.py:405: sigmoid(gate) > threshold, strict, frame included) or the frame cap
__device__ __forceinline__ bool slot_stops(const AdmitArgs &a, int j, int u, int f) {
    int cap = a.max_steps;
    if (a.cap_cur) cap = min(cap, a.cap_cur[j]);
    else if (a.caps) cap = min(cap, max(1, (int)a.caps[u]));
    if (f + 1 >= cap) return true;
    return !a.ignore_gate && sigmoidf_(a.out_t[(size_t)j * a.OL + a.M]) > a.thr;
}

__device__ void copy_rows(float *__restrict__ dst, const float *__restrict__ src, size_t n) {
    if ((((uintptr_t)dst | (uintptr_t)src) & 15) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (size_t i = threadIdx.x; i < n / 4; i += blockDim.x) d4[i] = s4[i];
        for (size_t i = n / 4 * 4 + threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    } else {
        for (size_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
    }
}

// one CTA per slot.  Step mode: write the slot's frame, apply the stop test, and let the slots that stop take queue entries.
// Head mode: no step ran; the idle slots take queue entries.  Either way the freed slots take entries next, next + 1, ...
// in slot order, and every CTA recomputes all S decisions to find its own prefix count.
__global__ void __launch_bounds__(ADMIT_THREADS) k_gate_admit(const AdmitArgs a) {
    pdl_trigger();
    pdl_wait();
    const int me = blockIdx.x, tid = threadIdx.x;
    const int next = a.next_cur[0];
    int n_free = 0, n_before = 0, n_active = 0;
    for (int base = 0; base < a.S; base += blockDim.x) {
        const int j = base + tid;
        bool act = false, fr = false;
        if (j < a.S) {
            const int u = a.utt_cur[j];
            act = u >= 0;
            fr = a.head ? !act : act && slot_stops(a, j, u, a.frame_cur[j]);
        }
        n_free += __syncthreads_count(fr);
        n_before += __syncthreads_count(fr && j < me);
        n_active += __syncthreads_count(act);
    }
    const int u = a.utt_cur[me], f = a.frame_cur[me];
    const bool stop = !a.head && u >= 0 && slot_stops(a, me, u, f);
    const int n_stop = a.head ? 0 : n_free;
    if (!a.head && a.ch_utt) {
        // 1. (session) the slot's row of this step in the chunk buffers
        const size_t k = (size_t)a.step * a.S + me;
        if (tid == 0) { a.ch_utt[k] = u; a.ch_frame[k] = u >= 0 ? f : 0; a.ch_last[k] = stop ? 1 : 0; }
        if (u >= 0) {
            const float *row = a.out_t + (size_t)me * a.OL;
            for (int m = tid; m <= a.M; m += blockDim.x) a.ch_frames[k * (a.M + 1) + m] = row[m];
            if (a.ch_align) {
                const float *al = a.align_t + (size_t)me * a.N;
                for (int n = tid; n < a.N; n += blockDim.x) a.ch_align[k * a.N + n] = al[n];
            }
        }
    } else if (!a.head && u >= 0) {
        // 1. the slot's frame f of utterance u
        const float *row = a.out_t + (size_t)me * a.OL;
        for (int m = tid; m < a.M; m += blockDim.x) a.mel_out[((size_t)u * a.M + m) * a.max_steps + f] = row[m];
        if (tid == 0) a.gate_out[(size_t)u * a.max_steps + f] = row[a.M];
        if (a.align_out) {
            const float *al = a.align_t + (size_t)me * a.N;
            float *dst = a.align_out + ((size_t)u * a.max_steps + f) * a.N;
            for (int n = tid; n < a.N; n += blockDim.x) dst[n] = al[n];
        }
        // 2. its frame count
        if (stop && tid == 0) a.n_frames[u] = f + 1;
    }
    // 3. admission
    int nu = u, nf = a.head ? f : f + 1, ncap = a.cap_cur ? a.cap_cur[me] : 0;
    if (a.head ? u < 0 : stop) {
        const int q = next + n_before;
        nu = q < a.U ? q : -1;
        nf = 0;
        if (nu >= 0) {
            const size_t e = a.cap ? (size_t)(q % a.cap) : (size_t)q;
            __syncthreads();           // the output row read above is zeroed below
            copy_rows(a.mem_slot + (size_t)me * a.N * a.E, a.memory + e * a.N * a.E, (size_t)a.N * a.E);
            copy_rows(a.pm_slot + (size_t)me * a.N * a.D, a.pmq + e * a.N * a.D, (size_t)a.N * a.D);
            if (tid == 0) a.len_slot[me] = a.lengths ? a.lengths[e] : (int64_t)a.N;
            ncap = a.caps ? max(1, (int)a.caps[e]) : a.max_steps;
            // the go frame: only the mel columns, the gate column of every slot is read by every CTA
            for (int m = tid; m < a.M; m += blockDim.x) a.out_t[(size_t)me * a.OL + m] = 0.f;
            for (int z = 0; z < a.nzero; ++z) {
                float *r = a.zero[z] + (size_t)me * a.zero_w[z];
                for (int i = tid; i < a.zero_w[z]; i += blockDim.x) r[i] = 0.f;
            }
            for (int z = 0; z < a.nimg; ++z) {
                __nv_bfloat16 *p = a.img[z] + (size_t)me * 64;
                for (int i = tid; i < a.img_k[z]; i += blockDim.x) p[(size_t)(i >> 6) * a.npad * 64 + (i & 63)] = __float2bfloat16(0.f);
            }
        }
    }
    if (tid == 0) {
        a.utt_nxt[me] = nu;
        a.frame_nxt[me] = nu >= 0 ? nf : 0;
        if (a.cap_nxt) a.cap_nxt[me] = ncap;
        if (me == 0) {
            // 4. active slots after this step, for the host poll
            const int admitted = min(n_free, max(0, a.U - next));
            a.next_nxt[0] = next + admitted;
            a.flags[0] = n_active - n_stop + admitted;
            if (a.cap) { a.flags[1] = next + admitted; a.flags[2] += n_stop; }
            if (a.bar) *a.bar = a.bar_value;
        }
    }
}

// slots 0 .. S-1 start with utterances 0 .. S-1; slots past the queue are idle (memory zero, length N)
__global__ void k_slot_start(int S, int U, int N, const int64_t *__restrict__ lengths, int64_t *__restrict__ len_slot,
                             int *__restrict__ st) {
    for (int s = blockIdx.x * blockDim.x + threadIdx.x; s < S; s += gridDim.x * blockDim.x) {
        st[s] = s < U ? s : -1;
        st[2 * S + s] = 0;
        len_slot[s] = (s < U && lengths) ? lengths[s] : (int64_t)N;
        if (s == 0) st[4 * S] = S < U ? S : U;
    }
}

// admission resets a slot's rows of the plan's recurrent state (InferPlan::state)
inline void admit_state(AdmitArgs &a, const InferPlan &P, float *s) {
    P.state(s, [&](float *p, int width) { a.zero[a.nzero] = p; a.zero_w[a.nzero] = width; ++a.nzero; },
            [&](bf16 *p, int kpad) { a.img[a.nimg] = p; a.img_k[a.nimg] = kpad; ++a.nimg; a.npad = P.Lb.NPAD; });
}

int infer_continuous(const InferPlan &P, const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths,
                     int U, int max_steps, const int32_t *frame_caps, float gate_threshold, int ignore_gate, uint64_t seed,
                     int row_offset, float *mel_out, float *gate_out, float *align_out, int32_t *n_frames, long long *steps_run,
                     int win_back, int win_fwd, float *s, cudaStream_t st) {
    const Dims &d = P.d;
    const int S = P.B, N = P.N;
    const ContL C(d, P.total, U, N, S);
    int *flags = P.flags(s), *state = (int *)(s + C.ST);
    int64_t *len_slot = (int64_t *)(s + C.LEN);
    float *mem_slot = s + C.MEM;
    const size_t SNE = (size_t)S * N * d.E;

    // processed memory of the whole queue, in launches of exactly S x N rows (the static call's row count, so every row
    // gets the bits the static call computes); the last launch is padded through the slot-memory buffer
    for (int u0 = 0; u0 < U; u0 += S) {
        const int n = U - u0 < S ? U - u0 : S;
        const float *src = memory + (size_t)u0 * N * d.E;
        if (n < S) {
            GVX_CUDA(cudaMemsetAsync(mem_slot, 0, SNE * sizeof(float), st));
            GVX_CUDA(cudaMemcpyAsync(mem_slot, src, (size_t)n * N * d.E * sizeof(float), cudaMemcpyDeviceToDevice, st));
            src = mem_slot;
        }
        GVX_TRY(run_processed_memory(d, w, src, S, N, s + C.PMQ + (size_t)u0 * N * d.D, st));
    }
    const int first = U < S ? U : S;
    GVX_CUDA(cudaMemsetAsync(mem_slot, 0, SNE * sizeof(float), st));
    GVX_CUDA(cudaMemcpyAsync(mem_slot, memory, (size_t)first * N * d.E * sizeof(float), cudaMemcpyDeviceToDevice, st));
    GVX_CUDA(cudaMemcpyAsync(s + P.PM, s + C.PMQ, (size_t)S * N * d.D * sizeof(float), cudaMemcpyDeviceToDevice, st));
    k_slot_start<<<grid_for(S), 256, 0, st>>>(S, U, N, mem_lengths, len_slot, state);
    GVX_LAUNCHED(1);
    k_fill_i32<<<grid_for(U), 256, 0, st>>>(n_frames, U, 0, 0);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());

    // recurrent state: zero at the start, and per row at every admission (k_gate_admit)
    GVX_TRY(P.reset(s, st));
    GVX_CUDA(cudaMemsetAsync(s + P.OUT, 0, (size_t)2 * S * d.OL * sizeof(float), st));     // the previous-frame ring: go frames
    AdmitArgs a;
    memset(&a, 0, sizeof(a));
    admit_state(a, P, s);
    a.align_t = s + C.ALIGN;
    a.memory = memory; a.pmq = s + C.PMQ; a.lengths = mem_lengths; a.caps = frame_caps;
    a.mem_slot = mem_slot; a.pm_slot = s + P.PM; a.len_slot = len_slot;
    a.mel_out = mel_out; a.gate_out = gate_out; a.align_out = align_out; a.n_frames = n_frames; a.flags = flags;
    a.thr = gate_threshold;
    a.ignore_gate = ignore_gate; a.S = S; a.U = U; a.N = N; a.E = d.E; a.D = d.D; a.M = d.M; a.OL = d.OL; a.max_steps = max_steps;
    InferStepArgs io;
    memset(&io, 0, sizeof(io));
    io.memory = mem_slot; io.lengths = len_slot;
    io.align_t = s + C.ALIGN; io.align_bstride = N;
    io.seed = seed; io.row_offset = row_offset;
    io.win_back = win_back; io.win_fwd = win_fwd;

    // every slot runs at most ceil(U/S) utterances' worth of max_steps before the queue is empty and its last one stops
    const long long bound = (long long)((U + S - 1) / S) * max_steps;
    long long t = 0;
    int host_running = first;
    for (; t < bound; ++t) {
        const int p = (int)(t & 1);
        int *utt = state + p * S, *frame = state + 2 * S + p * S;
        io.t = (int)t;
        io.row_frame = frame; io.row_id = utt;
        io.prev = s + P.OUT + (size_t)(p ^ 1) * S * d.OL;
        io.out_t = s + P.OUT + (size_t)p * S * d.OL;
        // full dependency on the previous step's k_gate_admit: kernels of the chain read the lengths and prefetch the
        // processed memory before griddepcontrol.wait, and an admission rewrites both
        pdl_barrier_next();
        GVX_TRY(P.step(w, packed, s, io, st));
        a.out_t = io.out_t;
        a.utt_cur = utt; a.frame_cur = frame; a.next_cur = state + 4 * S + p;
        a.utt_nxt = state + (p ^ 1) * S; a.frame_nxt = state + 2 * S + (p ^ 1) * S; a.next_nxt = state + 4 * S + (p ^ 1);
        GVX_CUDA(launch_pdl(k_gate_admit, dim3(S), dim3(ADMIT_THREADS), 0, st, a));
        GVX_LAUNCHED(1);
        GVX_CUDA(cudaGetLastError());
        if ((t + 1) % GVX_STOP_POLL == 0 || t + 1 == bound) {
            GVX_CUDA(cudaMemcpyAsync(&host_running, flags, sizeof(int), cudaMemcpyDeviceToHost, st));
            GVX_CUDA(cudaStreamSynchronize(st));
            if (host_running == 0) { ++t; break; }
        }
    }
    *steps_run = t;
    GVX_CHECK(host_running == 0, "continuous inference: slots still active after the step bound");
    return 0;
}

}  // namespace gvx

extern "C" {

size_t gvx_dec_infer_continuous_workspace_bytes(const gvx_dims *d, int U, int N, int slots) {
    using namespace gvx;
    if (check_dims(d) || U <= 0 || N <= 0 || slots <= 0) return 0;
    const InferPlan P(*d, slots, N, 2);
    if (P.bf && check_bf16_dims(P.d, slots)) return 0;
    return ContL(P.d, P.total, U, N, slots).total * sizeof(float);
}

int gvx_dec_infer_continuous_windowed(const gvx_dims *dd, const gvx_weights *w, const void *packed, const float *memory,
                                      const int64_t *mem_lengths, int U, int N, int slots, int max_steps, const int32_t *frame_caps,
                                      float gate_threshold, int ignore_gate, uint64_t seed, int row_offset, float *mel_out,
                                      float *gate_out, float *align_out, int32_t *n_frames, long long *steps_run, int att_backward,
                                      int att_forward, void *workspace, void *stream) {
    using namespace gvx;
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed && memory && mel_out && gate_out && n_frames && steps_run && workspace, "null argument");
    GVX_CHECK(U > 0 && N > 0 && slots > 0 && max_steps > 0, "U, N, slots, max_steps must be positive");
    GVX_TRY(check_window(att_backward, att_forward));
    GVX_TRY(latch_check());
    const InferPlan P(*dd, slots, N, 2);
    if (P.bf) GVX_TRY(check_bf16_dims(P.d, slots));
    cudaStream_t st = (cudaStream_t)stream;
    float *s = (float *)workspace;
    return infer_call(P, s, true, seed, st, "gvx_dec_infer_continuous", [&] {
        return infer_continuous(P, w, (const float *)packed, memory, mem_lengths, U, max_steps, frame_caps, gate_threshold, ignore_gate,
                                seed, row_offset, mel_out, gate_out, align_out, n_frames, steps_run, att_backward, att_forward, s, st);
    });
}

int gvx_dec_infer_continuous(const gvx_dims *dd, const gvx_weights *w, const void *packed, const float *memory,
                             const int64_t *mem_lengths, int U, int N, int slots, int max_steps, const int32_t *frame_caps,
                             float gate_threshold, int ignore_gate, uint64_t seed, int row_offset, float *mel_out, float *gate_out,
                             float *align_out, int32_t *n_frames, long long *steps_run, void *workspace, void *stream) {
    return gvx_dec_infer_continuous_windowed(dd, w, packed, memory, mem_lengths, U, N, slots, max_steps, frame_caps, gate_threshold,
                                             ignore_gate, seed, row_offset, mel_out, gate_out, align_out, n_frames, steps_run, 0, 0,
                                             workspace, stream);
}

}  // extern "C"
