"""Decoder sessions against re-batched continuous calls for requests that arrive over time (one GPU).

Workload: the utterances and frame caps of profiles/continuous_bench.py (BASELINE configs[3]'s token counts 75-150, gate
ignored, each utterance stopping at a cap of tokens x U[4.5, 7.5]), the first --utterances of its arrival order, arriving
on a seeded Poisson schedule measured in decoder steps.  Loads are fractions of what 64 slots sustain given the mean cap
(64 / mean cap utterances per step).

  rebatch   whenever the decoder is free, one Decoder.inference_continuous call (64 slots) over everything that has
            arrived; every frame of the call is returned when the call ends;
  session   one Decoder.session (64 slots): utterances are submitted at step-call boundaries and step(16) returns the
            frames of every call;
  up-front  the whole queue submitted before the first step, against one inference_continuous call on the same queue:
            what cutting the decode into step calls of 16 costs.

The clock is the decoder step: while the decoder has nothing to do it jumps to the next arrival (no waiting on the host).
A frame counts as returned when the call that returns it ends.  Latencies from arrival to first and to last returned frame
are given in steps and in seconds; seconds are steps times the arm's measured time per decoder step.  Utterances/s and
steps/s are over the time the decoder was busy.  The device name and power limit are read in the same run.
Usage: python profiles/session_bench.py [--utterances 1024] [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from continuous_bench import BATCH, MAX_STEPS, device_line, workload  # noqa: E402

CHUNK = 16
LOADS = (0.60, 0.85, 1.00)


def arrivals(caps, load, seed=29):
    """Poisson arrivals, in decoder steps, at `load` x the rate 64 slots sustain"""
    rate = load * BATCH / float(caps.double().mean())
    gaps = np.random.default_rng(seed).exponential(1.0 / rate, size=len(caps))
    return np.floor(np.cumsum(gaps)).astype(np.int64)


def rebatch_arm(dec, mem, ln, caps_dev, arr):
    U, clock, i, busy, first, last = len(arr), 0, 0, 0.0, np.zeros(len(arr)), np.zeros(len(arr))
    steps = 0
    while i < U:
        clock = max(clock, int(arr[i]))
        j = int(np.searchsorted(arr, clock, side="right"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dec.inference_continuous(mem[i:j], ln[i:j], slots=BATCH, max_decoder_steps=MAX_STEPS, frame_caps=caps_dev[i:j],
                                 ignore_gate=True, return_alignments=False)
        torch.cuda.synchronize()
        busy += time.perf_counter() - t0
        clock += dec.last_steps_run
        steps += dec.last_steps_run
        first[i:j] = last[i:j] = clock
        i = j
    return first, last, steps, busy


def session_arm(dec, mem, ln, caps_dev, arr, up_front=False):
    U = len(arr)
    sess = dec.session(mem.shape[1], slots=BATCH, capacity=U, max_decoder_steps=MAX_STEPS, ignore_gate=True,
                       return_alignments=False)
    first, last = np.full(U, -1.0), np.zeros(U)
    clock, i, busy, done = 0, 0, 0.0, 0
    torch.cuda.synchronize()
    while done < U:
        if not (sess.active or sess.pending) and i < U:
            clock = max(clock, int(arr[i]))
        j = U if up_front else int(np.searchsorted(arr, clock, side="right"))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if j > i:
            sess.submit(mem[i:j], ln[i:j], caps_dev[i:j])
            i = j
        before = sess.steps_run
        chunks, fin = sess.step(CHUNK)
        torch.cuda.synchronize()
        busy += time.perf_counter() - t0
        clock += sess.steps_run - before
        for u in chunks:
            if first[u] < 0:
                first[u] = clock
        for u in fin:
            last[u] = clock
        done += len(fin)
    return first, last, sess.steps_run, busy


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utterances", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import genvox_b200
    from genvox_b200 import _native
    if not torch.cuda.is_available():
        raise SystemExit("session_bench.py measures on the GPU; no CUDA device here")
    dev = torch.device("cuda:0")
    lib = _native.load()
    torch.manual_seed(0)
    from bench import decoder_dims
    dec = genvox_b200.Decoder(**decoder_dims()).to(dev).eval()
    memory, tokens, caps = workload(dev)
    perm = torch.randperm(len(caps), generator=torch.Generator().manual_seed(13))[:args.utterances]
    mem, ln, cp = memory[perm.to(dev)].contiguous(), tokens[perm.to(dev)].contiguous(), caps[perm].contiguous()
    cp_dev = cp.to(dev)
    info = device_line()
    print(json.dumps(info), flush=True)
    U = len(cp)
    results = []

    def record(precision, load, arm, arr, first, last, steps, busy, launches):
        per_step = busy / steps
        lat1, latn = first - arr, last - arr
        row = {"precision": precision, "load": load, "arm": arm, "utterances": U, "decoder_steps": int(steps),
               "busy_seconds": busy, "utterances_per_s": U / busy, "steps_per_s": steps / busy,
               "launches_per_step": launches / steps}
        for name, lat in (("first", lat1), ("last", latn)):
            for q in (50, 99):
                v = float(np.percentile(lat, q))
                row[f"{name}_p{q}_steps"] = v
                row[f"{name}_p{q}_s"] = v * per_step
        results.append(row)
        print(json.dumps(row), flush=True)

    def timed(fn):
        c0 = lib.gvx_launch_count()
        out = fn()
        return out + (lib.gvx_launch_count() - c0,)

    for precision in ("fp32", "bf16"):
        dec.precision = precision
        warm = np.zeros(2 * BATCH, dtype=np.int64)                       # warm-up of every arm's code path
        rebatch_arm(dec, mem[:2 * BATCH], ln[:2 * BATCH], cp_dev[:2 * BATCH], warm)
        session_arm(dec, mem[:2 * BATCH], ln[:2 * BATCH], cp_dev[:2 * BATCH], warm)
        for load in LOADS:
            arr = arrivals(cp, load)
            for arm, fn in (("rebatch", rebatch_arm), ("session", session_arm)):
                first, last, steps, busy, launches = timed(lambda: fn(dec, mem, ln, cp_dev, arr))
                record(precision, load, arm, arr, first, last, steps, busy, launches)
        zero = np.zeros(U, dtype=np.int64)
        first, last, steps, busy, launches = timed(lambda: rebatch_arm(dec, mem, ln, cp_dev, zero))
        record(precision, "up-front", "inference_continuous", zero, first, last, steps, busy, launches)
        first, last, steps, busy, launches = timed(lambda: session_arm(dec, mem, ln, cp_dev, zero, up_front=True))
        record(precision, "up-front", "session", zero, first, last, steps, busy, launches)
        genvox_b200.check_device_errors()
    print(f"\n{info['device']}, power limit / max SM clock: {info['power_limit_and_max_sm_clock']}; {U} utterances, "
          f"mean cap {float(cp.double().mean()):.1f} frames")
    print(f"{'prec':5} {'load':>8} {'arm':21} {'first p50/p99 steps':>20} {'last p50/p99 steps':>19} {'first p50/p99 s':>16} "
          f"{'last p50/p99 s':>15} {'utt/s':>7} {'steps/s':>8} {'launch/step':>11}")
    for r in results:
        print(f"{r['precision']:5} {str(r['load']):>8} {r['arm']:21} {r['first_p50_steps']:9.0f}/{r['first_p99_steps']:<10.0f} "
              f"{r['last_p50_steps']:9.0f}/{r['last_p99_steps']:<9.0f} {r['first_p50_s']:7.3f}/{r['first_p99_s']:<8.3f} "
              f"{r['last_p50_s']:7.3f}/{r['last_p99_s']:<7.3f} {r['utterances_per_s']:7.1f} {r['steps_per_s']:8.0f} "
              f"{r['launches_per_step']:11.3f}")
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"device": info, "results": results}, fh, indent=1)


if __name__ == "__main__":
    main()
