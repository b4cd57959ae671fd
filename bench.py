#!/usr/bin/env python
"""bench.py — throughput of the Tacotron2 decoder recurrence (the hot path, SURVEY.md §8) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[2] — data-parallel TRAINING, batch 64 per GPU,
150 tokens, 800x80 mel frames — one "step" is Tacotron2.train_step (tacotron2.py:515-522) restricted to
the decoder: zero_grad, Decoder.forward, loss, BPTT, [gradient all-reduce], clip_grad_norm_, Adam.
`value` = mel-frames/s with inputs resident in HBM, CUDA-event timed, max over ranks;
`e2e`   = the same step through genvox_b200.Decoder with HOST (pinned) inputs: H2D of memory/mel/gate
          and a D2H read of the loss inside the timed region;
`infer` = BASELINE.json configs[1] (batch 64, 1000 fixed decoder steps, fp32) in decoder steps/s, with its own e2e
          (host memory in, mel out) and weight-streaming roofline;
`roofline` for the dominant kernel of the step, from CUDA events the library records around every
phase launch during one extra profiled step (gvx_profile_*);
`cpu_baseline` = the UNMODIFIED reference Decoder (oracle/_ref, staged by oracle/build_ref.py; "kind": "reference") - or the
          oracle port when that tree is absent ("port") - on the host cores, on a bounded sample of the same workload;
`gpu_torch_baseline` = the same reference modules executed by stock PyTorch on the SAME GPU (fp32 and bf16 autocast; training
          and the batched decode loop): the number north_star asks to beat.
--impl reference times the CPU implementation alone (rank 0 only under torchrun), on this arm's config.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TRAIN = dict(B=64, N=150, T=int(os.environ.get("GVX_BENCH_T", "800")))     # BASELINE.json configs[2] (per GPU); the env
                                                                           # override is for debugging runs only
INFER = dict(B=64, N=150, steps=1000)     # BASELINE.json configs[1]
CPU_SAMPLE_T = 64                         # frames of the training workload the CPU legs run per step (fixed costs of a
                                          # step - zero_grad, clip, Adam over 18 M parameters - are then < 5 % of it)
GPU_TORCH_SAMPLE_T = 100                  # frames per step of the stock-PyTorch-on-GPU baseline
METRIC = "Tacotron2 train mel-frames/s"
UNIT = "mel-frames/s"


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], source="measured")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


def decoder_dims():
    return dict(n_mels=80, encoder_embedding_dim=512, decoder_rnn_dim=1024, prenet_dim=256, max_decoder_steps=1000,
                gate_threshold=0.5, p_attention_dropout=0.1, p_decoder_dropout=0.1, attention_rnn_dim=1024,
                attention_dim=128, attention_location_n_filters=32, attention_location_kernel_size=31)


def synthetic_batch(torch, B, N, T, rank=0):
    """Synthetic decoder inputs of the named shape (SURVEY.md §8d): encoder outputs, teacher-forcing mels
    (input and target), gate target 1 at the last frame (models/tts/__init__.py:53), full lengths."""
    g = torch.Generator().manual_seed(1 + rank)
    memory = 0.5 * torch.randn(B, N, 512, generator=g)
    mel = torch.randn(B, 80, T, generator=g)
    gate = torch.zeros(B, T)
    gate[:, -1] = 1.0
    lengths = torch.full((B,), N, dtype=torch.int64)
    return memory, mel, gate, lengths


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------ baseline legs (reference / oracle port)
def workload_config(world, precision, B, N, T):
    return {"workload": f"BASELINE configs[2]: decoder train step (fwd + loss + BPTT + allreduce + clip + Adam), "
                        f"batch {B}/GPU, {N} tokens, {T}x80 mel frames, "
                        + ("bf16 tcgen05 gate GEMMs with fp32 accumulation, fp32 pointwise/attention"
                           if precision == "bf16" else "fp32 arithmetic"),
            "global_batch": world * B, "parallelism": f"dp{world}",
            "l2": "per-step working set (stash + workspace, several GB) is far larger than the 126 MB L2"}


def _baseline_decoder(device):
    """The UNMODIFIED reference Decoder (models/tts/tacotron2.py:258-414, imported from /root/reference or from the copy
    oracle/build_ref.py staged under oracle/_ref) with the same init as the GPU arm; None when no reference tree exists."""
    import torch
    from oracle import ref_import as R
    if not R.reference_available():
        return None
    ref = R.import_reference()
    torch.manual_seed(0)
    return ref.Decoder(**decoder_dims()).to(device).train()


def _train_step_fn(torch, dec, P, opt, memory, mel, gate, lengths, autocast=None):
    """One decoder train step (tacotron2.py:515-522 restricted to the decoder) of the reference module `dec`, or of the oracle
    port over the parameter dict `P` when the reference tree is absent."""
    from genvox_b200.training import decoder_loss
    from oracle import decoder_oracle as O
    params = list(dec.parameters()) if dec is not None else list(P.values())

    def step(i):
        opt.zero_grad(set_to_none=True)
        ctx = torch.autocast("cuda", dtype=autocast) if autocast is not None else __import__("contextlib").nullcontext()
        with ctx:
            if dec is not None:
                m, g, _ = dec(memory, mel, lengths)
            else:
                m, g, _ = O.forward_teacher(P, memory, mel, lengths, seed=123 + i, training=True)
        loss, _, _ = decoder_loss(m.float(), g.float(), mel, gate)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        return loss

    return step


def cpu_train_leg(steps, warmup, sample_T=CPU_SAMPLE_T):
    """The reference's own CPU implementation of the same train step on the host cores, on a bounded sample of the workload:
    the full batch (64 x 150 tokens) but `sample_T` teacher-forced frames per step."""
    import torch
    import genvox_b200
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    B, N = TRAIN["B"], TRAIN["N"]
    dec = _baseline_decoder("cpu")
    P = None
    if dec is None:
        torch.manual_seed(0)
        cont = genvox_b200.Decoder(**decoder_dims())          # parameter container only: same init as the GPU arm
        P = {k: v.detach().clone().requires_grad_(True) for k, v in cont.named_parameters()}
    opt = torch.optim.Adam(list(dec.parameters()) if dec is not None else list(P.values()), lr=1e-3, weight_decay=1e-6)
    memory, mel, gate, lengths = synthetic_batch(torch, B, N, sample_T)
    step = _train_step_fn(torch, dec, P, opt, memory, mel, gate, lengths)
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    what = ("the unmodified reference Decoder (models/tts/tacotron2.py via oracle/_ref)" if dec is not None
            else "oracle/decoder_oracle.py (port: no reference tree staged)")
    return dict(value=B * sample_T / dt, unit=UNIT, cores=cores, threads=torch.get_num_threads(),
                kind="reference" if dec is not None else "port",
                sample=f"{what}, train step (fwd+loss+BPTT+clip+Adam) on CPU fp32, B={B}, N={N}, {sample_T} of "
                       f"{TRAIN['T']} frames per step, {steps} timed steps after {warmup} warm-up",
                ms_per_step=dt * 1e3)


def torch_gpu_legs(dev, steps=2, warmup=1, sample_T=GPU_TORCH_SAMPLE_T, infer_steps=100):
    """Stock PyTorch on the SAME GPU: the reference modules (eager kernels: cuBLAS GEMMs, ATen LSTM-cell pointwise, cuDNN
    conv, autograd BPTT) on a bounded sample of the training workload - fp32 as the reference runs it, and under bf16
    autocast - plus the batched decode loop (initialize_decoder_states / prenet / decode driven for B rows, as the public
    inference is B = 1 only).  This is the "cuDNN/PyTorch GPU path" north_star asks to beat."""
    import torch
    import torch.nn.functional as F
    import genvox_b200
    from oracle import decoder_oracle as O
    B, N = TRAIN["B"], TRAIN["N"]
    out = {"device": torch.cuda.get_device_name(dev), "sample": f"B={B}, N={N}, {sample_T} of {TRAIN['T']} frames per train step; "
                                                               f"{infer_steps} of {INFER['steps']} decode steps"}
    memory, mel, gate, lengths = (t.to(dev) for t in synthetic_batch(torch, B, N, sample_T))
    # the port runs on the GPU here with torch's dropout and a device mask; the CPU leg after this one needs the originals
    oracle_fns = O.philox_dropout, O.get_mask_from_lengths
    try:
        for name, ac in (("train_fp32", None), ("train_bf16_autocast", torch.bfloat16)):
            dec = _baseline_decoder(dev)
            P = None
            if dec is None:
                torch.manual_seed(0)
                cont = genvox_b200.Decoder(**decoder_dims())
                P = {k: v.detach().clone().to(dev).requires_grad_(True) for k, v in cont.named_parameters()}
                O.philox_dropout = lambda x, p, on, *a, **k: F.dropout(x, p, on)
                O.get_mask_from_lengths = lambda lengths, max_len=None: (
                    torch.arange(max_len if max_len is not None else int(lengths.max()), device=dev)[None, :] >= lengths.to(dev)[:, None])
            opt = torch.optim.Adam(list(dec.parameters()) if dec is not None else list(P.values()), lr=1e-3, weight_decay=1e-6)
            step = _train_step_fn(torch, dec, P, opt, memory, mel, gate, lengths, autocast=ac)
            for i in range(warmup):
                step(i)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            for i in range(steps):
                step(warmup + i)
            torch.cuda.synchronize(dev)
            dt = (time.perf_counter() - t0) / steps
            out[name] = {"mel_frames_per_s": B * sample_T / dt, "ms_per_step": dt * 1e3, "kind": "reference" if dec is not None else "port"}
            del opt, step, dec, P
    finally:
        O.philox_dropout, O.get_mask_from_lengths = oracle_fns
    dec = _baseline_decoder(dev)
    if dec is not None:
        dec.eval()
        mem_i = memory[:INFER["B"]]
        for name, ac in (("infer_fp32", None), ("infer_bf16_autocast", torch.bfloat16)):
            def run(n):
                with torch.no_grad(), (torch.autocast("cuda", dtype=ac) if ac is not None else __import__("contextlib").nullcontext()):
                    dec.initialize_decoder_states(mem_i, mask=None)
                    x = mem_i.new_zeros(mem_i.shape[0], 80)
                    for _ in range(n):
                        m, _, _ = dec.decode(dec.prenet(x))
                        x = m.float()
            run(10)
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            run(infer_steps)
            torch.cuda.synchronize(dev)
            dt = (time.perf_counter() - t0) / infer_steps
            out[name] = {"decoder_steps_per_s": 1.0 / dt, "us_per_step": dt * 1e6, "kind": "reference"}
    return out


def run_reference(args, rank):
    if rank != 0:
        return
    leg = cpu_train_leg(args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, args.precision, TRAIN["B"], TRAIN["N"], TRAIN["T"]),
            "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ roofline accounting
def slot_rooflines(phases, B, N, T, pk, precision):
    """One roofline entry per profiler slot; the algorithmic FLOPs / bytes of an entry are those of the kernels THAT slot
    brackets (DESIGN.md section 5 lists them).  Tensor-bound entries: 2 * MACs of the contractions in the slot over the slot's
    device time against the measured sustained bf16 rate; HBM-bound entries (the attention chains): SURVEY.md 8(d)'s
    per-step attention bytes over the chain's time per step against the measured copy bandwidth."""
    H = A = 1024
    E, D, P, M, F = 512, 128, 256, 80, 32
    Kd, Ka, Kp = A + E + H, P + E + A, H + E
    TB = float(T) * B
    fused = phases.get("attention", {}).get("launches") == 1          # persistent chains: ONE launch for all T steps
    roofs = {}

    def tensor(name, flops, kernels, burst=False):
        if name not in phases or phases[name]["ms"] <= 0:
            return
        ach = flops / (phases[name]["ms"] * 1e-3) / 1e12
        # a slot that is ONE short library-shaped GEMM is a kernel timed alone: the burst figure is its peak (B200_PROFILING.md);
        # the persistent chains run for milliseconds: sustained
        peak = pk["tf_burst"] if burst else pk["tf_sustained"]
        roofs[name] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                       "traffic": None, "avg_us": phases[name]["avg_us"], "us_per_step": 1e3 * phases[name]["ms"] / T,
                       "launches": phases[name]["launches"], "algorithmic_flops": flops, "kernels": kernels,
                       "peak_source": pk["source"] + (" (bf16 burst)" if burst else " (bf16 sustained)")
                                      + ("" if precision == "bf16" else "; fp32 mode runs FFMA")}

    def hbm(name, bytes_per_step, kernels, note=None):
        if name not in phases or phases[name]["ms"] <= 0:
            return
        per_step_us = 1e3 * phases[name]["ms"] / T
        ach = bytes_per_step / (per_step_us * 1e-6) / 1e9
        roofs[name] = {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                       "traffic": None, "avg_us": phases[name]["avg_us"], "us_per_step": per_step_us,
                       "launches": phases[name]["launches"], "algorithmic_bytes_per_step": bytes_per_step, "kernels": kernels,
                       "peak_source": pk["source"]}
        if note:
            roofs[name]["note"] = note

    if fused:
        tensor("att_lstm", 2.0 * TB * P * 4 * A, "time-batched GEMM: prenet part of the attention-LSTM gates, all frames", burst=True)
        hbm("attention", B * N * (E * 2.0 + D * 4.0) + B * N * 4.0, "k_att_chain_fwd (attention LSTM + query + attention, all T steps)",
            "latency-bound persistent chain (2 grid barriers + 2 exchanges per step); operands L2 resident")
        tensor("dec_lstm_input_gemm", 2.0 * TB * (A + E) * 4 * H, "time-batched GEMM: input part of the decoder-LSTM gates", burst=True)
        tensor("dec_lstm", 2.0 * TB * H * 4 * H, "k_lstm_chain_fwd (recurrent part, all T steps)")
        tensor("output", 2.0 * TB * (M + 1) * Kp, "time-batched GEMM: mel / gate projections")
        tensor("bwd_dec_pointwise", 2.0 * TB * H * 4 * H, "k_lstm_chain_bwd (decoder-LSTM BPTT, all T steps)")
        tensor("bwd_dec_gemm", 2.0 * TB * (A + E) * 4 * H, "time-batched GEMM: d [h_att | ctx] from the decoder-LSTM input", burst=True)
        hbm("bwd_attention", B * N * (E * 2.0 + D * 2.0) + B * N * 4.0, "k_att_chain_bwd (attention-chain BPTT, all T steps)",
            "latency-bound persistent chain (3 inter-SM exchanges per step); bf16 memory + bf16 tanh stash read, d e written")
        tensor("bwd_time_batched", 2.0 * TB * (4 * H * Kd + 4 * A * Ka + 4 * A * P + D * A + (M + 1) * Kp + 2 * P * P + P * M)
               + 2.0 * TB * N * (D * F + 2 * F * 31) + 4.0 * B * N * D * E,
               "weight-gradient / prenet GEMMs, attention-parameter reductions, d memory")
    else:
        for name, Kc in (("dec_lstm", Kd), ("att_lstm", Ka), ("bwd_dec_gemm", Kd), ("bwd_att_gemm", Ka)):
            tensor(name, 2.0 * TB * Kc * 4 * H, "gate GEMM of every step (per-step launch chain)")
        for name in ("attention", "bwd_attention"):
            hbm(name, B * N * (E + D) * 4.0 + B * N * 4.0, "per-step attention kernel")
    return roofs


# ------------------------------------------------------------------------------------ GPU arm
DUMP_MAX_ELEMS = 1 << 20      # per array; larger ones are sampled, so that a dump stays near 36 MB (at most 64 MB)


def dump_outputs(out_dir, dec, loss, grad_norm):
    """--dump-outputs: what the last timed train step hands its caller - the loss and the gradient norm it returns, and the
    decoder's parameters and (clipped) gradients as the step leaves them - as float32 <name>.npy files in `out_dir`.  An array
    of more than DUMP_MAX_ELEMS elements is stored flattened at a fixed, seeded sample of positions (the same in every run),
    so that two builds can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, "grad_norm": grad_norm}
    for k, p in dec.named_parameters():
        arrays[f"param.{k}"] = p
        arrays[f"grad.{k}"] = p.grad
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > DUMP_MAX_ELEMS:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def _stage(rank, msg):
    if os.environ.get("GVX_BENCH_TRACE"):
        print(f"[rank {rank}] {time.strftime('%H:%M:%S')} {msg}", file=sys.stderr, flush=True)


def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import genvox_b200
    from genvox_b200 import _native
    from genvox_b200.training import decoder_train_step, make_optimizer

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device (the product has no CPU path; use --impl reference for the CPU leg)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _native.load()
    B, N, T = TRAIN["B"], TRAIN["N"], TRAIN["T"]
    K, Wm = args.steps, max(args.warmup, 3)

    torch.manual_seed(0)                                   # identical init on every rank
    dec = genvox_b200.Decoder(**decoder_dims()).to(dev).train()
    dec.precision = args.precision
    dec.dropout_row_offset = rank * B                      # ranks draw the rows of one global batch
    opt = make_optimizer(dec)
    memory_h, mel_h, gate_h, lengths_h = (t.pin_memory() for t in synthetic_batch(torch, B, N, T, rank))
    memory, mel, gate, lengths = (t.to(dev) for t in (memory_h, mel_h, gate_h, lengths_h))
    group = dist.group.WORLD if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step_resident(sync_gradients=True):
        return decoder_train_step(dec, opt, memory, mel, gate, lengths, group=group, sync_gradients=sync_gradients)

    loss_h = torch.zeros(1).pin_memory()

    def step_e2e():
        m = memory_h.to(dev, non_blocking=True)
        x = mel_h.to(dev, non_blocking=True)
        g = gate_h.to(dev, non_blocking=True)
        le = lengths_h.to(dev, non_blocking=True)
        loss, _ = decoder_train_step(dec, opt, m, x, g, le, group=group)
        loss_h.copy_(loss.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(loss_h[0])

    # ---- value: inputs resident in HBM
    _stage(rank, "setup done")
    for i in range(Wm):
        step_resident()
        if os.environ.get("GVX_BENCH_SYNC"):
            torch.cuda.synchronize()
        _stage(rank, f"warm-up step {i} enqueued")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if sampler:
        sampler.start()
    launches0 = lib.gvx_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    host_t0 = time.perf_counter()
    for _ in range(K):
        loss, grad_norm = step_resident()
    host_enqueue_ms = (time.perf_counter() - host_t0) * 1e3 / K      # host time to ENQUEUE a step (no sync inside)
    e1.record()
    barrier()
    launches = lib.gvx_launch_count() - launches0
    clocks = sampler.stop() if sampler else None
    _stage(rank, "timed region done")
    if args.dump_outputs and rank == 0:          # before the e2e steps below change the parameters again
        dump_outputs(args.dump_outputs, dec, loss, grad_norm)
    ms = max_over_ranks(e0.elapsed_time(e1)) / K
    value = world * B * T / (ms * 1e-3)
    final_loss = float(loss)

    # ---- e2e: host buffers, H2D + D2H inside the timed region
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        step_e2e()
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3) / K
    _stage(rank, "e2e done")
    h2d = sum(t.numel() * t.element_size() for t in (memory_h, mel_h, gate_h, lengths_h))
    e2e = {"value": world * B * T / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms,
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(world, args.precision, B, N, T),
            "e2e": e2e, "gpu_launches": int(launches), "final_loss": final_loss, "host_enqueue_ms_per_step": host_enqueue_ms}
    if clocks is not None:
        line["clocks"] = clocks
    gs = (C.c_ulonglong * 4)()
    lib.gvx_graph_stats(gs)
    line["cuda_graphs"] = {"eager_calls": int(gs[0]), "captured": int(gs[1]), "replays": int(gs[2]), "failed_captures": int(gs[3])}

    if rank == 0:
        # ---- one extra, profiled step: per-phase device time from CUDA events around every launch
        lib.gvx_profile_reset()
        lib.gvx_profile_enable(1)
        step_resident(sync_gradients=False)      # rank 0 alone: no collective in this extra step
        torch.cuda.synchronize()
        lib.gvx_profile_enable(0)
        phases, slot = {}, 0
        while True:
            name = lib.gvx_profile_slot_name(slot)
            if name is None:
                break
            tot, cnt = C.c_double(0), C.c_longlong(0)
            lib.gvx_profile_read(slot, C.byref(tot), C.byref(cnt))
            if cnt.value:
                phases[name.decode()] = {"ms": tot.value, "launches": cnt.value, "avg_us": 1e3 * tot.value / cnt.value}
            slot += 1
        line["phases_ms"] = {k: round(v["ms"], 3) for k, v in phases.items()}
        pk = peaks()
        roofs = slot_rooflines(phases, B, N, T, pk, args.precision)
        tpath = os.path.join(ROOT, "profiles", "traffic_r2.json")
        if os.path.isfile(tpath):          # DRAM bytes per launch from the committed ncu --set full capture
            with open(tpath) as fh:
                traffic = json.load(fh)
            for k, r in roofs.items():
                if k in traffic:
                    r["traffic"] = traffic[k]["dram_bytes_per_launch"]
                    r["traffic_note"] = f'ncu {traffic[k]["kernel"]}, {traffic[k]["launch"]}'
        if roofs:
            dominant = max(roofs, key=lambda k: phases[k]["ms"])
            line["roofline"] = dict(roofs[dominant], kernel=dominant)
            line["roofline_all"] = roofs
        # ---- inference, BASELINE configs[1] (fp32 as the config states; bf16 reported beside it)
        dec.eval()
        mem_i = memory[:INFER["B"]]
        mem_ih = memory_h[:INFER["B"]].clone().pin_memory()
        infer = {"workload": f"BASELINE configs[1]: batch {INFER['B']}, {INFER['N']} tokens, {INFER['steps']} fixed "
                             "decoder steps (gate ignored)"}
        step_weights = 18.19e6                       # parameters every decoder step touches (SURVEY.md 8d)
        for prec in ("fp32", "bf16"):
            dec.precision = prec
            for _ in range(2):
                dec.inference(mem_i, ignore_gate=True, max_decoder_steps=INFER["steps"])
            torch.cuda.synchronize()
            e0.record()
            reps = 3
            for _ in range(reps):
                dec.inference(mem_i, ignore_gate=True, max_decoder_steps=INFER["steps"])
            e1.record()
            torch.cuda.synchronize()
            ims = e0.elapsed_time(e1) / reps
            # end to end: encoder memory from pinned host memory, mel frames back to the host
            t0 = time.perf_counter()
            for _ in range(reps):
                m_i, _, _ = dec.inference(mem_ih.to(dev, non_blocking=True), ignore_gate=True, max_decoder_steps=INFER["steps"])
                mel_host = m_i.cpu()
            e2e_ims = (time.perf_counter() - t0) * 1e3 / reps
            wbytes = step_weights * (4.0 if prec == "fp32" else 2.0)
            ach = wbytes / (ims * 1e-3 / INFER["steps"]) / 1e9
            infer[prec] = {"decoder_steps_per_s": INFER["steps"] / (ims * 1e-3),
                           "mel_frames_per_s": INFER["B"] * INFER["steps"] / (ims * 1e-3), "us_per_step": 1e3 * ims / INFER["steps"],
                           "e2e": {"decoder_steps_per_s": INFER["steps"] / (e2e_ims * 1e-3), "h2d_bytes": mem_ih.numel() * 4,
                                   "d2h_bytes": mel_host.numel() * 4},
                           "roofline": {"bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                                        "algorithmic_bytes_per_step": wbytes, "traffic": None,
                                        "note": "weight streaming: every step reads all recurrent / projection weights once "
                                                "(they do not fit on chip in one kernel); SURVEY.md 8(d)"}}
        dec.precision = args.precision
        infer["decoder_steps_per_s"] = infer["fp32"]["decoder_steps_per_s"]       # headline: the config's own precision
        line["infer"] = infer
        dec.train()
        if world == 1 and not args.no_gpu_torch:
            # free this arm's memory first: the eager reference keeps ~(86 KB + 1168 N) bytes per sample-step for autograd
            del dec, opt
            torch.cuda.empty_cache()
            line["gpu_torch_baseline"] = torch_gpu_legs(dev)
            t = line["gpu_torch_baseline"]
            t["ours_over_torch"] = {"train_bf16": value / t["train_bf16_autocast"]["mel_frames_per_s"],
                                    "train_vs_fp32_eager": value / t["train_fp32"]["mel_frames_per_s"]}
            if "infer_fp32" in t:
                t["ours_over_torch"]["infer_fp32"] = infer["fp32"]["decoder_steps_per_s"] / t["infer_fp32"]["decoder_steps_per_s"]
                t["ours_over_torch"]["infer_bf16"] = infer["bf16"]["decoder_steps_per_s"] / t["infer_bf16_autocast"]["decoder_steps_per_s"]
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = {k: v for k, v in cpu_train_leg(2, 1).items() if k != "ms_per_step"}
        line["library"] = {"path": os.path.relpath(_native.library_path(), ROOT), "fresh": bool(_native.library_is_fresh())}
        print(json.dumps(line), flush=True)


def run_infer_sharded(args, rank, world, local_rank):
    """BASELINE configs[3]: 4096 synthetic utterances sharded over the GPUs of the box (contiguous shards, NO collective on the
    data path), decoded in batches of 64 by `Decoder.inference`; gate-stopped with at most 1000 steps as the config says, and
    - because a random-init gate fires (or never fires) on the first steps - the gate-ignored variant beside it."""
    import torch
    import torch.distributed as dist
    import genvox_b200
    from genvox_b200.training import shard_rows
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    U, Bt, steps = int(os.environ.get("GVX_BENCH_UTTERANCES", "4096")), 64, INFER["steps"]
    lo, hi = shard_rows(U, rank, world)
    torch.manual_seed(0)
    dec = genvox_b200.Decoder(**decoder_dims()).to(dev).eval()
    dec.precision = args.precision
    g = torch.Generator().manual_seed(7)
    lengths_all = torch.sort(torch.randint(75, 151, (U,), generator=g), descending=True).values      # token counts, longest first
    batches = []
    for b0 in range(lo, hi, Bt):
        ln = lengths_all[b0:min(b0 + Bt, hi)]
        gb = torch.Generator().manual_seed(1000 + b0)
        mem = 0.5 * torch.randn(len(ln), int(ln.max()), 512, generator=gb)
        for r, n in enumerate(ln.tolist()):
            mem[r, n:] = 0
        batches.append((mem.to(dev), ln.to(dev)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    res = {}
    for variant, ignore in (("gate_stopped", False), ("gate_ignored", True)):
        for mem, ln in batches[:1]:
            dec.inference(mem, memory_lengths=ln, ignore_gate=ignore, max_decoder_steps=steps)          # warm-up
        barrier()
        t0 = time.perf_counter()
        frames = 0
        nsteps = 0
        for mem, ln in batches:
            m, _, _ = dec.inference(mem, memory_lengths=ln, ignore_gate=ignore, max_decoder_steps=steps)
            frames += int(dec.last_n_frames.sum().item())
            nsteps += m.shape[2]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        genvox_b200.check_device_errors()
        t = torch.tensor([dt, float(frames), float(nsteps)], dtype=torch.float64, device=dev)
        if world > 1:
            tm = t.clone()
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            dt = float(tm[0].item())
        res[variant] = {"utterances_per_s": U / dt, "mel_frames_per_s": float(t[1].item()) / dt,
                        "decoder_steps_per_s_per_gpu": float(t[2].item()) / world / dt, "seconds": dt}
    if rank == 0:
        print(json.dumps({"metric": "Tacotron2 sharded batched inference", "value": res["gate_ignored"]["utterances_per_s"],
                          "unit": "utterances/s", "n_gpus": world, "higher_is_better": True, "scaling": "strong",
                          "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
                          "config": {"workload": f"BASELINE configs[3]: {U} synthetic utterances (75-150 tokens) sharded over {world} "
                                                 f"GPU(s), batches of {Bt}, max {steps} decoder steps; no data-path collective"},
                          "variants": res}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-gpu-torch", action="store_true", help="skip the stock-PyTorch-on-GPU baseline legs")
    ap.add_argument("--mode", choices=["train", "infer_sharded"], default="train",
                    help="train: BASELINE configs[2] (the contract's line); infer_sharded: configs[3], utterances sharded over the GPUs")
    ap.add_argument("--precision", choices=["bf16", "fp32"], default="bf16",
                    help="arithmetic of the recurrent GEMMs (BASELINE configs[2] is bf16; fp32 = parity mode)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (loss, gradient norm, the decoder's "
                         "parameters and gradients) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "train"):
        ap.error("--dump-outputs needs --impl ours --mode train")

    # watchdog: a run that has not finished after 10 minutes (the default run takes about one) dumps every thread's Python
    # stack and exits instead of hanging its caller; GVX_BENCH_TRACE=1 adds per-stage progress lines on stderr
    import faulthandler
    faulthandler.dump_traceback_later(int(os.environ.get("GVX_BENCH_TRACE_AFTER", "600")), exit=True)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1 and "RANK" not in os.environ:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29531"),
               os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))
    try:
        if args.mode == "infer_sharded":
            run_infer_sharded(args, rank, world, local_rank)
        else:
            run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
