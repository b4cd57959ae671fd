// genvox_b200 — training: the per-precision plan of a teacher-forced forward and its BPTT, and their entry points.
// The forward and the backward see the precision, and in bf16 the chains they run, only through TrainPlan: its stash and
// backward layouts, the seed slot and one BfTrainPath.  The forward writes the stash in the formats of that path; the
// backward of a plan with the same path reads them.
#pragma once
#include "gvx_bf16_api.cuh"
#include "gvx_bwd.cuh"
#include "gvx_graph.cuh"

namespace gvx {

// A train step of B rows, N memory frames and T decoder frames, in the layouts of its precision: StashL / BwdL in fp32,
// StashBfL / BwdBfL in bf16.
struct TrainPlan {
    Dims d;
    bool bf;
    int B, N, T;
    StashL Sf;
    BwdL Wf;
    StashBfL Sb;
    BwdBfL Wb;
    size_t stash_total, bwd_total, SEED;     // in floats; SEED: the stash slot of the dropout seed {lo, hi}
    BfTrainPath path;                        // bf16 chains of both passes; decided only when `run` (it asks the device what fits)

    TrainPlan(const gvx_dims &dd, int rows, int n, int t, bool run)
        : d(dd), bf(dd.precision == GVX_BF16), B(rows), N(n), T(t), Sf(d, B, N, T), Wf(d, B, N, T), Sb(d, B, N, T), Wb(d, B, N, T),
          stash_total(bf ? Sb.total : Sf.total), bwd_total(bf ? Wb.total : Wf.total), SEED(bf ? Sb.SEED : Sf.SEED),
          path(bf && run ? bf_train_path(d, B, N) : BfTrainPath{}) {}

    uint32_t *seed_slot(const void *stash) const { return reinterpret_cast<uint32_t *>((float *)const_cast<void *>(stash) + SEED); }

    int fwd(const gvx_weights *w, const float *packed, const float *memory, const float *mel_in, const int64_t *mem_lengths,
            uint64_t seed, int training, int row_offset, float *mel_out, float *gate_out, float *align_out, float *s,
            cudaStream_t st) const {
        if (bf)
            return train_fwd_bf16(d, path, Sb, w, packed, memory, mel_in, mem_lengths, B, N, T, seed, training, row_offset, mel_out,
                                  gate_out, align_out, s, st);
        return train_fwd_fp32(d, Sf, w, packed, memory, mel_in, mem_lengths, B, N, T, seed, training, row_offset, mel_out, gate_out,
                              align_out, s, st);
    }

    int bwd(const gvx_weights *w, const float *packed, const float *memory, const int64_t *mem_lengths, uint64_t seed, int training,
            int row_offset, const float *d_mel, const float *d_gate, const float *d_align, const float *s, float *x,
            const gvx_grads *g, float *d_memory, cudaStream_t st) const {
        GVX_CHECK(d.F <= 64 && d.D <= 512, "backward supports loc_filters <= 64 and att_dim <= 512");
        if (bf)
            return train_bwd_bf16(d, path, Sb, Wb, w, packed, memory, mem_lengths, B, N, T, seed, training, row_offset, d_mel, d_gate,
                                  d_align, s, x, g, d_memory, st);
        return train_bwd_fp32(d, Sf, Wf, w, packed, memory, mem_lengths, B, N, T, seed, training, row_offset, d_mel, d_gate, d_align,
                              s, x, g, d_memory, st);
    }
};

// The frame of both training entry points: the dropout seed into the plan's seed slot (the backward stores the value its
// forward stored), then the body through the CUDA-graph cache under `key`, with g_seed_ptr at that slot (the dropout of its
// kernels reads the seed there, so a captured graph outlives it).
template <class Body>
int train_call(const TrainPlan &P, const void *stash, uint64_t seed, const std::string &key, cudaStream_t user, Body &&body) {
    uint32_t *slot = P.seed_slot(stash);
    GVX_TRY(put_seed(slot, seed, user));
    g_seed_ptr = slot;
    const int rc = run_cached(key, user, body);
    g_seed_ptr = nullptr;
    return rc;
}

}  // namespace gvx

extern "C" {

size_t gvx_dec_stash_bytes(const gvx_dims *d, int B, int N, int T) {
    using namespace gvx;
    if (check_dims(d) || B <= 0 || N <= 0 || T <= 0) return 0;
    return TrainPlan(*d, B, N, T, false).stash_total * sizeof(float);
}

size_t gvx_dec_bwd_workspace_bytes(const gvx_dims *d, int B, int N, int T) {
    using namespace gvx;
    if (check_dims(d) || B <= 0 || N <= 0 || T <= 0) return 0;
    return TrainPlan(*d, B, N, T, false).bwd_total * sizeof(float);
}

int gvx_dec_train_fwd(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                      const float *mel_in, const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training,
                      int row_offset, float *mel_out, float *gate_out, float *align_out, void *stash_, void *stream) {
    using namespace gvx;
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_ && memory && mel_in && mel_out && gate_out && align_out && stash_, "null argument");
    GVX_CHECK(B > 0 && N > 0 && T > 0, "B, N, T must be positive");
    GVX_TRY(latch_check());
    const TrainPlan P(*dd, B, N, T, true);
    KeyBuilder kb;
    kb.add((int)1).add(*dd).add(*w).add(packed_).add(memory).add(mel_in).add(mem_lengths).add(B).add(N).add(T).add(training)
        .add(row_offset).add(mel_out).add(gate_out).add(align_out).add(stash_);
    return train_call(P, stash_, seed, kb.k, (cudaStream_t)stream, [&](cudaStream_t st) {
        return P.fwd(w, (const float *)packed_, memory, mel_in, mem_lengths, seed, training, row_offset, mel_out, gate_out, align_out,
                     (float *)stash_, st);
    });
}

int gvx_dec_train_bwd(const gvx_dims *dd, const gvx_weights *w, const void *packed_, const float *memory,
                      const int64_t *mem_lengths, int B, int N, int T, uint64_t seed, int training,
                      int row_offset, const float *d_mel, const float *d_gate, const float *d_align,
                      const void *stash_, void *workspace, const gvx_grads *g, float *d_memory, void *stream) {
    using namespace gvx;
    GVX_TRY(check_dims(dd));
    GVX_CHECK(w && packed_ && memory && d_mel && d_gate && stash_ && workspace && g && d_memory, "null argument");
    GVX_CHECK(B > 0 && N > 0 && T > 0, "B, N, T must be positive");
    GVX_TRY(latch_check());
    const TrainPlan P(*dd, B, N, T, true);
    KeyBuilder kb;
    kb.add((int)2).add(*dd).add(*w).add(packed_).add(memory).add(mem_lengths).add(B).add(N).add(T).add(training).add(row_offset)
        .add(d_mel).add(d_gate).add(d_align).add(stash_).add(workspace).add(*g).add(d_memory);
    return train_call(P, stash_, seed, kb.k, (cudaStream_t)stream, [&](cudaStream_t st) {
        return P.bwd(w, (const float *)packed_, memory, mem_lengths, seed, training, row_offset, d_mel, d_gate, d_align,
                     (const float *)stash_, (float *)workspace, g, d_memory, st);
    });
}

}  // extern "C"
