// genvox_b200 — continuous-batching inference: a queue of U utterances decoded through S fixed decoder slots.
//
// Static batching (gvx_dec_infer) runs every batch until its last row stops, so rows that stop early sit idle.  Here a slot
// whose utterance stops takes the next utterance of the queue on the device, before the next decoder step: k_gate_admit runs
// in the launch slot k_gate_check has in the static loop.  Per step it writes each slot's frame straight into its
// utterance's outputs, applies the stop test, admits and resets, and publishes the number of active slots for the host
// poll.  Admission is deterministic and uses no atomics: the slots that stop in the same step take queue entries in slot
// order, and every CTA recomputes all S stop decisions to find its own prefix count.
//
// Output identity: utterance u decodes bit-identically to row r of a static call with the same S rows, N, seed and
// precision, u in row r and dropout_row_offset = u + row_offset - r.  The slot's every piece of recurrent state is zeroed
// in the layout it lives in, its memory / processed memory / length are replaced, and the prenet draws its dropout at
// Philox (row u + row_offset, t = local frame) through the per-row row_frame / row_id arrays.
#pragma once
#include "gvx_bf16_api.cuh"

namespace gvx {

// ---- workspace: the static inference layout for S rows and a two-frame output ring (steps = 2), then this block
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

inline size_t continuous_base(const Dims &d, bool bf, int S, int N) {
    return bf ? InferBfL(d, S, N, 2).total : InferL(d, S, N, 2).total;
}

// the per-row recurrent state an admission zeroes, in the layout it lives in: fp32 h/c of both LSTMs, ctx, attention weights
// and cumulative weights; in bf16 mode the cell states, attention weights and the slot's rows of the tcgen05 operand images
inline void admit_state(AdmitArgs &a, const Dims &d, bool bf, const InferL &Lf, const InferBfL &Lb, float *s, int S, int N) {
    auto zrow = [&](float *p, int width) { a.zero[a.nzero] = p; a.zero_w[a.nzero] = width; ++a.nzero; };
    if (bf) {
        const BfGeom g(d);
        zrow(s + Lb.CA, d.A); zrow(s + Lb.CD, d.H); zrow(s + Lb.WPREV, N); zrow(s + Lb.CUM, N);
        bf16 *XAI = (bf16 *)(s + Lb.XAI), *XDI = (bf16 *)(s + Lb.XDI);
        a.img[0] = XAI; a.img[1] = XAI + Lb.xai_stride; a.img_k[0] = a.img_k[1] = g.Kpa;
        a.img[2] = XDI; a.img[3] = XDI + Lb.xdi_stride; a.img_k[2] = a.img_k[3] = g.Kpd;
        a.img[4] = (bf16 *)(s + Lb.XPI); a.img_k[4] = g.Kpp;
        a.nimg = 5;
        a.npad = Lb.NPAD;
    } else {
        zrow(s + Lf.HA, d.A); zrow(s + Lf.HA + (size_t)S * d.A, d.A); zrow(s + Lf.CA, d.A);
        zrow(s + Lf.HD, d.H); zrow(s + Lf.HD + (size_t)S * d.H, d.H); zrow(s + Lf.CD, d.H);
        zrow(s + Lf.CTX, d.E); zrow(s + Lf.WPREV, N); zrow(s + Lf.CUM, N);
    }
}

int infer_continuous(const gvx_dims *dd, const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths,
                     int U, int N, int S, int max_steps, const int32_t *frame_caps, float gate_threshold, int ignore_gate,
                     uint64_t seed, int row_offset, float *mel_out, float *gate_out, float *align_out, int32_t *n_frames,
                     long long *steps_run, float *s, cudaStream_t st) {
    const Dims d(*dd);
    const bool bf = dd->precision == GVX_BF16;
    if (bf) GVX_TRY(check_bf16_dims(d, S));
    const InferL Lf(d, S, N, 2);
    const InferBfL Lb(d, S, N, 2);
    const ContL C(d, continuous_base(d, bf, S, N), U, N, S);
    const size_t PM = bf ? Lb.PM : Lf.PM, OUT = bf ? Lb.OUT : Lf.OUT, FLAGS = bf ? Lb.FLAGS : Lf.FLAGS;
    int *flags = (int *)(s + FLAGS), *state = (int *)(s + C.ST);
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
    GVX_CUDA(cudaMemcpyAsync(s + PM, s + C.PMQ, (size_t)S * N * d.D * sizeof(float), cudaMemcpyDeviceToDevice, st));
    k_slot_start<<<grid_for(S), 256, 0, st>>>(S, U, N, mem_lengths, len_slot, state);
    GVX_LAUNCHED(1);
    k_fill_i32<<<grid_for(U), 256, 0, st>>>(n_frames, U, 0, 0);
    GVX_LAUNCHED(1);
    GVX_CUDA(cudaGetLastError());

    // recurrent state: zero at the start, and per row at every admission (k_gate_admit)
    AdmitArgs a;
    memset(&a, 0, sizeof(a));
    admit_state(a, d, bf, Lf, Lb, s, S, N);
    if (bf) {
        const BfGeom g(d);
        GVX_CUDA(cudaMemsetAsync(s + Lb.ERR, 0, 64 * sizeof(float), st));
        GVX_CUDA(cudaMemsetAsync(a.img[0], 0, 2 * Lb.xai_stride * sizeof(bf16), st));
        GVX_CUDA(cudaMemsetAsync(a.img[2], 0, 2 * Lb.xdi_stride * sizeof(bf16), st));
        GVX_CUDA(cudaMemsetAsync(a.img[4], 0, (size_t)g.Kpp * Lb.NPAD * sizeof(bf16), st));
    }
    for (int z = 0; z < a.nzero; ++z) GVX_CUDA(cudaMemsetAsync(a.zero[z], 0, (size_t)S * a.zero_w[z] * sizeof(float), st));
    GVX_CUDA(cudaMemsetAsync(s + OUT, 0, (size_t)2 * S * d.OL * sizeof(float), st));     // the previous-frame ring: go frames
    GVX_CUDA(cudaMemsetAsync(flags, 0, 32 * sizeof(int), st));       // [0] active slots; [32..33] hold the dropout seed
    GVX_CUDA(cudaMemsetAsync(flags + 40, 0, 2 * sizeof(int), st));   // [40] prenet grid barrier, [41] its error word

    a.align_t = s + C.ALIGN;
    a.memory = memory; a.pmq = s + C.PMQ; a.lengths = mem_lengths; a.caps = frame_caps;
    a.mem_slot = mem_slot; a.pm_slot = s + PM; a.len_slot = len_slot;
    a.mel_out = mel_out; a.gate_out = gate_out; a.align_out = align_out; a.n_frames = n_frames; a.flags = flags;
    a.thr = gate_threshold;
    a.ignore_gate = ignore_gate; a.S = S; a.U = U; a.N = N; a.E = d.E; a.D = d.D; a.M = d.M; a.OL = d.OL; a.max_steps = max_steps;
    const bool fused_prenet = infer_prenet_fused_ok(d, S);

    // every slot runs at most ceil(U/S) utterances' worth of max_steps before the queue is empty and its last one stops
    const long long bound = (long long)((U + S - 1) / S) * max_steps;
    long long t = 0;
    int host_running = first;
    for (; t < bound; ++t) {
        const int p = (int)(t & 1);
        const float *prev = s + OUT + (size_t)(p ^ 1) * S * d.OL;
        float *out_t = s + OUT + (size_t)p * S * d.OL;
        int *utt = state + p * S, *frame = state + 2 * S + p * S;
        // full dependency on the previous step's k_gate_admit: kernels of the chain read the lengths and prefetch the
        // processed memory before griddepcontrol.wait, and an admission rewrites both
        pdl_barrier_next();
        if (bf) GVX_TRY(infer_step_bf16(d, w, packed, Lb, s, mem_slot, len_slot, S, N, seed, (int)t, 0, row_offset, frame, utt, prev,
                                        s + C.ALIGN, (long long)N, out_t, st));
        else GVX_TRY(infer_step(d, w, packed, Lf, s, mem_slot, len_slot, S, N, seed, (int)t, 0, row_offset, frame, utt, prev,
                                s + C.ALIGN, (long long)N, out_t, fused_prenet, st));
        a.out_t = out_t;
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
    const Dims dm(*d);
    const bool bf = d->precision == GVX_BF16;
    if (bf && check_bf16_dims(dm, slots)) return 0;
    return ContL(dm, continuous_base(dm, bf, slots, N), U, N, slots).total * sizeof(float);
}

int gvx_dec_infer_continuous(const gvx_dims *dd, const gvx_weights *w, const void *packed, const float *memory,
                             const int64_t *mem_lengths, int U, int N, int slots, int max_steps, const int32_t *frame_caps,
                             float gate_threshold, int ignore_gate, uint64_t seed, int row_offset, float *mel_out, float *gate_out,
                             float *align_out, int32_t *n_frames, long long *steps_run, void *workspace, void *stream) {
    using namespace gvx;
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed && memory && mel_out && gate_out && n_frames && steps_run && workspace, "null argument");
    GVX_CHECK(U > 0 && N > 0 && slots > 0 && max_steps > 0, "U, N, slots, max_steps must be positive");
    GVX_TRY(latch_check());
    cudaStream_t st = (cudaStream_t)stream;
    const Dims d(*dd);
    const bool bf = dd->precision == GVX_BF16;
    if (bf) GVX_TRY(check_bf16_dims(d, slots));
    const size_t flags_off = bf ? InferBfL(d, slots, N, 2).FLAGS : InferL(d, slots, N, 2).FLAGS;
    uint32_t *slot = reinterpret_cast<uint32_t *>((float *)workspace + flags_off) + 32;
    GVX_TRY(put_seed(slot, seed, st));
    g_seed_ptr = slot;
    int rc = infer_continuous(dd, w, (const float *)packed, memory, mem_lengths, U, N, slots, max_steps, frame_caps, gate_threshold,
                              ignore_gate, seed, row_offset, mel_out, gate_out, align_out, n_frames, steps_run, (float *)workspace, st);
    g_seed_ptr = nullptr;
    if (rc == 0 && bf)
        rc = check_tc_err_public(reinterpret_cast<int *>((float *)workspace + InferBfL(d, slots, N, 2).ERR), st,
                                 "gvx_dec_infer_continuous");
    if (rc == 0 && !bf)
        rc = check_tc_err_public(reinterpret_cast<int *>((float *)workspace + flags_off) + 41, st,
                                 "gvx_dec_infer_continuous (prenet barrier)");
    return rc;
}

}  // extern "C"
