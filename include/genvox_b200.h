/*
 * genvox_b200 — C ABI of the B200-native Tacotron2 decoder recurrence.
 *
 * Drop-in boundary for the ONE hot path of saiakarsh193/GenVox (SURVEY.md §8):
 * the decoder recurrence of models/tts/tacotron2.py.  The reference has no FFI (it is pure
 * Python/PyTorch); each entry point below cites the reference Python interface it replaces.
 * The host-side mirror (genvox_b200/decoder.py, class Decoder) binds these through ctypes;
 * INTEGRATION.md shows the binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates); the library
 *     keeps no device memory across calls;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no host sync
 *     (gvx_dec_infer with gate stop polls a device flag every GVX_STOP_POLL steps);
 *   - tensors are fp32, contiguous, in the reference's own layouts (stated per argument);
 *   - every function returns 0 on success, non-zero on error; gvx_last_error() returns the
 *     message for the calling thread.  There is no CPU fallback.
 *   - dropout uses the counter-based Philox4x32-10 stream defined in
 *     genvox_b200/csrc/gvx_common.cuh (host mirror: oracle/philox.py): keep iff
 *     philox(counter=(j>>2, row+row_offset, t, site), key=seed)[j&3] >= floor(p * 2^32).
 */
#ifndef GENVOX_B200_H
#define GENVOX_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GVX_ABI_VERSION 1
#define GVX_STOP_POLL 16

/* Constructor arguments of the reference Decoder, models/tts/tacotron2.py:259-273
 * (defaults: configs/models.py:10-33).  All feature dims must be multiples of 4. */
typedef struct gvx_dims {
    int32_t n_mels;            /* 80  */
    int32_t enc_dim;           /* encoder_embedding_dim, 512 */
    int32_t att_rnn_dim;       /* 1024 */
    int32_t dec_rnn_dim;       /* 1024 */
    int32_t prenet_dim;        /* 256 */
    int32_t att_dim;           /* 128 */
    int32_t loc_filters;       /* attention_location_n_filters, 32 */
    int32_t loc_kernel;        /* attention_location_kernel_size, 31 (odd) */
    float p_att_dropout;       /* 0.1 */
    float p_dec_dropout;       /* 0.1 */
    int32_t precision;         /* GVX_FP32: fp32 FFMA everywhere (parity mode, BASELINE configs[0],[1]);
                                  GVX_BF16: gate / query / projection GEMMs on tcgen05 with bf16 operands and fp32
                                  accumulation, pointwise math, cell state and attention in fp32 (configs[2],[4]);
                                  needs dims % 8 == 0, rnn dims % 32 == 0 and at most 128 rows per call */
} gvx_dims;
#define GVX_FP32 0
#define GVX_BF16 1

/* Decoder parameters in state_dict layout (SURVEY.md §8b), row-major [out, in]:
 * names are the reference's `decoder.*` keys. */
typedef struct gvx_weights {
    const float *prenet_w0;    /* prenet.layers.0.linear_layer.weight          [P, n_mels]      */
    const float *prenet_w1;    /* prenet.layers.1.linear_layer.weight          [P, P]           */
    const float *att_w_ih;     /* attention_rnn.weight_ih                      [4A, P+E]  i,f,g,o */
    const float *att_w_hh;     /* attention_rnn.weight_hh                      [4A, A]          */
    const float *att_b_ih;     /* attention_rnn.bias_ih                        [4A]             */
    const float *att_b_hh;     /* attention_rnn.bias_hh                        [4A]             */
    const float *query_w;      /* attention_layer.query_layer.linear_layer.weight   [D, A]      */
    const float *memory_w;     /* attention_layer.memory_layer.linear_layer.weight  [D, E]      */
    const float *v_w;          /* attention_layer.v.linear_layer.weight             [1, D]      */
    const float *loc_conv_w;   /* attention_layer.location_layer.location_conv.conv.weight [F, 2, K] */
    const float *loc_dense_w;  /* attention_layer.location_layer.location_dense.linear_layer.weight [D, F] */
    const float *dec_w_ih;     /* decoder_rnn.weight_ih                        [4H, A+E]        */
    const float *dec_w_hh;     /* decoder_rnn.weight_hh                        [4H, H]          */
    const float *dec_b_ih;     /* decoder_rnn.bias_ih                          [4H]             */
    const float *dec_b_hh;     /* decoder_rnn.bias_hh                          [4H]             */
    const float *proj_w;       /* linear_projection.linear_layer.weight        [n_mels, H+E]    */
    const float *proj_b;       /* linear_projection.linear_layer.bias          [n_mels]         */
    const float *gate_w;       /* gate_layer.linear_layer.weight               [1, H+E]         */
    const float *gate_b;       /* gate_layer.linear_layer.bias                 [1]              */
} gvx_weights;

/* Gradients, same shapes as gvx_weights; every buffer is fully overwritten. */
typedef struct gvx_grads {
    float *prenet_w0, *prenet_w1;
    float *att_w_ih, *att_w_hh, *att_b_ih, *att_b_hh;
    float *query_w, *memory_w, *v_w, *loc_conv_w, *loc_dense_w;
    float *dec_w_ih, *dec_w_hh, *dec_b_ih, *dec_b_hh;
    float *proj_w, *proj_b, *gate_w, *gate_b;
} gvx_grads;

int gvx_abi_version(void);
const char *gvx_last_error(void);

/* Device-side abort latch.  gvx_dec_train_fwd / gvx_dec_train_bwd never synchronise with the host, so a persistent or
 * tcgen05 kernel that aborted (a bounded wait timed out: the chain lost its co-resident CTAs, a pipeline stalled) cannot
 * fail the call that launched it.  Its error word is latched into pinned host memory by the last kernel of the call;
 * every later entry point returns non-zero once the latch is set, and this function returns the latched code
 * (entry * 1000 + wait code; 0 = none) without synchronising.  Call it after a stream / device synchronisation to
 * learn whether the outputs just produced are valid.  clear != 0 resets the latch.  (Python: genvox_b200.check_device_errors.) */
int gvx_device_error(int clear);

/* Number of SMs / device name the library sees on the current device (diagnostics). */
int gvx_device_info(int *sm_count, int *cc_major, int *cc_minor);

/* Accounting for bench.py: kernels launched by this library since load, and an optional phase
 * profiler.  When enabled every phase launch inside train_fwd / train_bwd / infer is bracketed by
 * CUDA events on the launching stream (slower; never on during a timed throughput run);
 * gvx_profile_read synchronises and returns the summed device time and the number of bracketed
 * launches of one slot; gvx_profile_slot_name returns NULL past the last slot. */
unsigned long long gvx_launch_count(void);
int gvx_profile_enable(int on);
int gvx_profile_reset(void);
int gvx_profile_read(int slot, double *total_ms, long long *launches);
const char *gvx_profile_slot_name(int slot);

/* CUDA-graph cache statistics: {calls run eagerly, graphs captured, graph replays, failed captures}.  The launch
 * sequence of train_fwd / train_bwd / fixed-step infer is captured the second time a call with identical arguments
 * (pointers, shapes, flags; the dropout seed lives in device memory) is seen and replayed afterwards. */
int gvx_graph_stats(unsigned long long *out4);

/* Repacked weights (gate rows interleaved per hidden unit, W_ih|W_hh concatenated, transposed
 * copies for backward).  Replaces nothing in the reference: it is the cached form of the
 * parameters owned by Decoder.__init__ (tacotron2.py:259-301).  Call again whenever the
 * parameters change (every optimizer step). */
size_t gvx_dec_packed_bytes(const gvx_dims *d);
int gvx_dec_pack_weights(const gvx_dims *d, const gvx_weights *w, void *packed, void *stream);

/* Sizes of the caller-allocated buffers for a [B rows, N tokens, T frames] call. */
size_t gvx_dec_stash_bytes(const gvx_dims *d, int B, int N, int T);      /* train_fwd -> train_bwd */
size_t gvx_dec_bwd_workspace_bytes(const gvx_dims *d, int B, int N, int T);
size_t gvx_dec_infer_workspace_bytes(const gvx_dims *d, int B, int N, int max_steps);

/* Teacher-forced forward: Decoder.forward, tacotron2.py:365-388 (prenet over all frames :373,
 * initialize_decoder_states :303-315, T x decode :333-363, parse_decoder_outputs :322-331).
 *   memory      [B, N, E]          encoder outputs
 *   mel_in      [B, n_mels, T]     decoder_inputs (batch["mel_padded"])
 *   mem_lengths [B] int64 or NULL  memory_lengths; tokens >= length get -inf energy (:125)
 *   training    LSTM-state dropout on/off (self.training, :341,:358); prenet dropout is always on (:143)
 *   mel_out [B, n_mels, T], gate_out [B, T], align_out [B, T, N]
 *   stash       gvx_dec_stash_bytes() bytes; consumed by gvx_dec_train_bwd */
int gvx_dec_train_fwd(const gvx_dims *d, const gvx_weights *w, const void *packed,
                      const float *memory, const float *mel_in, const int64_t *mem_lengths,
                      int B, int N, int T, uint64_t seed, int training, int row_offset,
                      float *mel_out, float *gate_out, float *align_out,
                      void *stash, void *stream);

/* Backward through time: what loss.backward() (tacotron2.py:520) does to the graph built by
 * Decoder.forward.  d_align may be NULL (the reference's loss never uses alignments, :598-615).
 *   d_mel [B, n_mels, T], d_gate [B, T], d_align [B, T, N] or NULL
 *   grads: all decoder parameters; d_memory [B, N, E] (overwritten) */
int gvx_dec_train_bwd(const gvx_dims *d, const gvx_weights *w, const void *packed,
                      const float *memory, const int64_t *mem_lengths,
                      int B, int N, int T, uint64_t seed, int training, int row_offset,
                      const float *d_mel, const float *d_gate, const float *d_align,
                      const void *stash, void *workspace,
                      const gvx_grads *grads, float *d_memory, void *stream);

/* Batched autoregressive inference: Decoder.inference, tacotron2.py:390-414, generalised to
 * B >= 1 rows (the reference loop is B = 1, :405).  Per row the frame count is the first
 * step whose sigmoid(gate) > gate_threshold (strict, frame included, :405) or max_steps
 * (:407); decoding continues until every row has stopped (ignore_gate: always max_steps).
 *   mel_out [B, n_mels, max_steps], gate_out [B, max_steps], align_out [B, max_steps, N]
 *   n_frames [B] int32 (device), *steps_run (host) = number of decoder steps executed
 * Only the first *steps_run frames of the outputs are written. */
int gvx_dec_infer(const gvx_dims *d, const gvx_weights *w, const void *packed,
                  const float *memory, const int64_t *mem_lengths,
                  int B, int N, int max_steps, float gate_threshold, int ignore_gate,
                  uint64_t seed, int training, int row_offset,
                  float *mel_out, float *gate_out, float *align_out, int32_t *n_frames,
                  int *steps_run, void *workspace, void *stream);

/* Continuous batching: decode a queue of U utterances (all padded to N tokens) through `slots` decoder rows.  Slots start
 * with utterances 0 .. slots-1; when a slot's utterance stops, the slot takes the next utterance of the queue on the device
 * before the next decoder step (slots stopping in the same step take them in slot order), with its recurrent state zeroed.
 * Utterance u stops at the first frame whose sigmoid(gate) > gate_threshold (as gvx_dec_infer; not with ignore_gate) or
 * after cap[u] = min(max_steps, frame_caps[u]) frames.  Its prenet dropout at local frame f draws Philox row
 * u + row_offset, t = f.  Eval mode only (no LSTM-state dropout).  bf16 mode: slots <= 128.
 * Output identity: utterance u's frames 0 .. n_frames[u]-1 are bit-identical to row r of a gvx_dec_infer call with the same
 * slots rows, N, seed and precision, u in row r and row_offset' = u + row_offset - r; n_frames[u] is that row's stop step.
 *   memory [U, N, E]; mem_lengths [U] int64 or NULL; frame_caps [U] int32 or NULL
 *   mel_out [U, n_mels, max_steps], gate_out [U, max_steps], align_out [U, max_steps, N] or NULL, n_frames [U] int32
 *   *steps_run (host) = decoder steps executed (at most ceil(U / slots) * max_steps)
 * Only frames 0 .. n_frames[u]-1 of the outputs are written. */
size_t gvx_dec_infer_continuous_workspace_bytes(const gvx_dims *d, int U, int N, int slots);
int gvx_dec_infer_continuous(const gvx_dims *d, const gvx_weights *w, const void *packed,
                             const float *memory, const int64_t *mem_lengths, int U, int N, int slots,
                             int max_steps, const int32_t *frame_caps, float gate_threshold, int ignore_gate,
                             uint64_t seed, int row_offset,
                             float *mel_out, float *gate_out, float *align_out, int32_t *n_frames,
                             long long *steps_run, void *workspace, void *stream);

/* Decoder sessions: continuous batching for requests that arrive over time.  A session holds `slots` decoder rows and their
 * recurrent state in a caller-owned workspace, plus a ring of `capacity` queued utterances (all padded to N tokens).  The
 * caller submits utterances between calls (ids 0, 1, 2, ... in submission order) and steps the session for up to k decoder
 * steps at a time: at the head of a step call the idle slots take queued utterances in slot order; during the call a slot
 * whose utterance stops takes the next queued one on the device, as in gvx_dec_infer_continuous.  Every step call returns
 * the frames it decoded, tagged per (step, slot).  The session is this struct plus the workspace: the library keeps no
 * device memory across calls, and both are used on one stream.  Eval mode only.  bf16 mode: slots <= 128.
 * Output identity: utterance `id` decodes bit-identically to row r of a gvx_dec_infer call with the same slots rows, N,
 * seed and precision, id in row r and row_offset' = id + row_offset - r, whatever the submission times, the step counts per
 * call and the other slots were; its frame count is that row's stop step (as gvx_dec_infer_continuous, with frame cap
 * min(max_steps, frame_caps[id])). */
typedef struct gvx_session {
    /* set by the caller before gvx_dec_session_init */
    int32_t N, slots, capacity, max_steps, ignore_gate, with_alignments, row_offset;
    float gate_threshold;
    uint64_t seed;
    /* maintained by the library */
    long long steps_run;   /* decoder steps run over the session's life */
    long long submitted;   /* utterances submitted = the next id */
    long long admitted;    /* utterances taken into a slot, read back at the end of each step call */
    long long finished;    /* utterances whose last frame was returned, read back at the end of each step call */
    int32_t active;        /* slots holding an utterance, read back at the end of each step call */
    int32_t parity;        /* which half of the workspace's slot-state ping-pong is current */
    int32_t ready;         /* set by gvx_dec_session_init */
} gvx_session;

/* Workspace bytes of a session; 0 for bad dims, N, slots or capacity, or bf16 with slots > 128.  It grows by
 * N * (enc_dim + att_dim) * 4 + 12 bytes per ring entry. */
size_t gvx_dec_session_workspace_bytes(const gvx_dims *d, int N, int slots, int capacity);
/* Checks the caller-set fields of *s, zeroes the workspace (every slot idle), stores the seed and resets the counters. */
int gvx_dec_session_init(const gvx_dims *d, gvx_session *s, void *workspace, void *stream);
/* Appends k utterances (ids s->submitted .. s->submitted + k - 1) and computes their processed memory.
 *   memory [k, N, E]; lengths [k] int64 or NULL (all N); frame_caps [k] int32 or NULL (max_steps)
 * Refused: submitted + k - admitted > capacity, or an id + row_offset past 2^31 - 1.  Asynchronous on `stream`. */
int gvx_dec_session_submit(const gvx_dims *d, const gvx_weights *w, const void *packed, gvx_session *s,
                           const float *memory, const int64_t *lengths, const int32_t *frame_caps, int k,
                           void *workspace, void *stream);
/* Runs up to max_steps_this_call (>= 1) decoder steps; it ends early once no slot is active (the queue is then empty: it
 * only grows between calls, and the idle slots take from it at the head of every call).  A session with no active slot
 * and no queued utterance runs 0 steps and launches nothing.  For step i < *steps_run and slot j (row i * slots + j):
 *   utt[i][j]    int32: the utterance the slot decoded, -1 = idle (the other outputs of that row are not written)
 *   frame[i][j]  int32: its local frame index;  last[i][j] int8: 1 on its last frame (its frame count is frame + 1)
 *   frames[i][j] [n_mels + 1] floats: the [mel | gate] row;  align[i][j] [N] floats (when align is not NULL)
 * Buffers are [max_steps_this_call][slots][...] device arrays.  Synchronises with the host (the stop poll, every
 * GVX_STOP_POLL steps and at the end) and updates steps_run, admitted, finished and active. */
int gvx_dec_session_step(const gvx_dims *d, const gvx_weights *w, const void *packed, gvx_session *s, int max_steps_this_call,
                         float *frames, float *align, int32_t *utt, int32_t *frame, int8_t *last, int *steps_run,
                         void *workspace, void *stream);

/* ---- single-phase entry points (used by the parity tests to localise a failure) ---- */

/* The tcgen05 / TMEM / TMA gate-GEMM engine on its own: out[B, Mtot] = X[B, K] . W[Mtot, K]^T with both
 * operands rounded to bf16, fp32 accumulation, the K range split over KS CTAs (test hook; allocates). */
int gvx_test_tc_gemm(const float *W, const float *X, int B, int Mtot, int K, int KS, float *out, void *stream);

/* Test hook: the tcgen05 GEMM of the time-batched contractions (csrc/gvx_nt_gemm.cuh) on its own.  Replaces nothing in the
 * reference by itself: it is the engine behind every all-frames nn.Linear / nn.LSTMCell contraction and their autograd weight
 * gradients (tacotron2.py:340,:357,:361-362,:520).  mode 0: C[M,N] = A[M,K] . B[N,K]^T; mode 1: A is [K,M], B is [K,N] (transposed on
 * the device first: the weight-gradient path, K = frames).  fp32 device pointers, operands rounded to bf16, fp32 accumulate. */
int gvx_test_nt_gemm(const float *A, const float *B, int M, int N, int K, int mode, float *C, void *stream);
/* Timing hook (profiles/nt_gemm_bench.py): average device time in ms of `reps` launches of that GEMM on zero-filled operands. */
int gvx_bench_nt_gemm(int M, int N, int K, int reps, float *ms_out);

/* The persistent LSTM-chain kernels on their own (test hook; allocates): for t < T
 *   gates_t = pre_t + h_{t-1} . W_hh^T (h, W_hh rounded to bf16, fp32 accumulate), nn.LSTMCell pointwise part
 *   (tacotron2.py:357), carried-state dropout (:358, Philox site 3), h_{-1} = c_{-1} = 0.
 *   w_hh [4H, H] torch layout (rows i,f,g,o); pre [T, B, 4H] with columns 4*unit + gate;
 *   h_out [T, B, H] (dropped h, bf16-rounded); c_out [T+1, B, H]; gates_out [T, B, 4H] activations (4*unit + gate).
 *   If dh_ext [T, B, H] (gradient w.r.t. the dropped h_t from outside the chain) and dgates_out [T, B, 4H] are given,
 *   BPTT runs too and dgates_out receives d loss / d pre (bf16-rounded). */
int gvx_test_lstm_chain(const float *w_hh, const float *pre, int B, int T, int H, float p_drop, uint64_t seed,
                        int training, float *h_out, float *c_out, float *gates_out, const float *dh_ext,
                        float *dgates_out, void *stream);

/* Debug hook: when non-null, CTA 0 of the persistent chain kernels writes clock64 stamps per step into
 * device_buffer ([4][1024][32] int64: decoder-LSTM forward chain, backward chain, progress markers, fused attention chain).  Pass NULL to switch it off. */
int gvx_debug_timeline(void *device_buffer);

/* Debug hook: force a code path on (1), off (0) or back to its environment default (-1).  Options: "fused" (the
 * persistent attention chain, env GVX_FUSED), "persistent" (the persistent decoder-LSTM chains, env GVX_PERSISTENT).
 * The parity tests use it to compare the fused and the per-step paths on the same inputs. */
int gvx_debug_option(const char *name, int value);

/* Prenet.forward, tacotron2.py:140-144: frames [F, B, n_mels] -> out [F, B, P]; frame f uses
 * Philox t = t0 + f.  tmp: [F, B, P] scratch for the layer-0 output. */
int gvx_prenet_fwd(const gvx_dims *d, const gvx_weights *w, const float *frames, int F, int B,
                   uint64_t seed, int t0, int row_offset, float *tmp, float *out, void *stream);

/* One nn.LSTMCell step + state dropout (tacotron2.py:340-341 / :357-358).
 * which = 0 attention_rnn, 1 decoder_rnn.  x [B, in], h/c [B, hid]; outputs h_out (dropped),
 * c_out, and optionally the gate activations [B, 4*hid] in packed (unit-major) order. */
int gvx_lstm_step(const gvx_dims *d, const void *packed, int which, const float *x, const float *h,
                  const float *c, int B, uint64_t seed, int t, int training, int row_offset,
                  float *h_out, float *c_out, float *gates_out, void *stream);

/* Attention.forward (tacotron2.py:106-129) + cumulative update (:353) for one step.
 * h_att [B, A]; processed_memory [B, N, D]; w_prev/w_cum [B, N] are updated in place;
 * ctx_out [B, E], align_out [B, N]; q_tmp [B, D] scratch. */
int gvx_attention_step(const gvx_dims *d, const gvx_weights *w, const void *packed, const float *h_att, const float *memory,
                       const float *processed_memory, const int64_t *mem_lengths, int B, int N,
                       float *w_prev, float *w_cum, float *q_tmp, float *ctx_out, float *align_out,
                       void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GENVOX_B200_H */
