"""Static against continuous batching for inference on one GPU (Decoder.inference vs Decoder.inference_continuous).

Workload: BASELINE configs[3]'s utterances as bench.py --mode infer_sharded makes them (token counts 75-150 from
torch.Generator seed 7, memories per batch of 64 from seed 1000 + first row), both as one GPU's shard of 8 (512 utterances)
and all 4096 on one GPU.  Random-init weights cannot produce realistic gate stops, so the gate is ignored and every
utterance stops at a frame cap: frames = tokens x r with r ~ U[4.5, 7.5] per utterance (a plausible spread of speaking rate,
seeded), at most 1000.

  static      today's path: batches of 64 through Decoder.inference(ignore_gate=True, max_decoder_steps=max cap in the batch),
              each batch padded to its own longest utterance;
  continuous  one Decoder.inference_continuous call with 64 slots, every utterance padded to the longest of the queue.

Both in the queue order bench.py uses (sorted by token count, longest first) and in arrival order (a seeded shuffle); the
two arms alternate 3 times in one process.  Per arm: utterances/s, decoder steps, mel-frames/s, slot occupancy
(frames / (64 x steps)) and launches per decoder step (gvx_launch_count), in fp32 and bf16.  The device name and power
limit are read in the same run.  Usage: python profiles/continuous_bench.py [--reps 3] [--out FILE.json]
"""
import argparse
import heapq
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

U_ALL, BATCH, MAX_STEPS, SHARD = 4096, 64, 1000, 512


def workload(dev):
    g = torch.Generator().manual_seed(7)
    tokens = torch.sort(torch.randint(75, 151, (U_ALL,), generator=g), descending=True).values       # bench.py, longest first
    N = int(tokens.max())
    memory = torch.zeros(U_ALL, N, 512)
    for b0 in range(0, U_ALL, BATCH):
        ln = tokens[b0:b0 + BATCH]
        gb = torch.Generator().manual_seed(1000 + b0)
        mem = 0.5 * torch.randn(len(ln), int(ln.max()), 512, generator=gb)
        for r, n in enumerate(ln.tolist()):
            memory[b0 + r, :n] = mem[r, :n]
    rate = 4.5 + 3.0 * torch.rand(U_ALL, generator=torch.Generator().manual_seed(11))
    caps = torch.clamp((tokens.double() * rate.double()).floor().long(), 1, MAX_STEPS).to(torch.int32)
    return memory.to(dev), tokens.to(dev), caps


def predicted_steps(caps, slots=BATCH):
    """decoder steps from the stop steps alone: static = sum of batch maxima; continuous = refill on stop, in slot order"""
    c = caps.tolist()
    static = sum(max(c[i:i + slots]) for i in range(0, len(c), slots))
    heap = [(c[s], s) for s in range(min(slots, len(c)))]
    heapq.heapify(heap)
    for u in range(len(heap), len(c)):
        t, s = heapq.heappop(heap)
        heapq.heappush(heap, (t + c[u], s))
    end = max(t for t, _ in heap)
    return static, end


def device_line():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:        # the query is informational; the numbers below do not depend on it
        q = f"unavailable ({exc})"
    return {"device": name, "power_limit_and_max_sm_clock": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import genvox_b200
    from genvox_b200 import _native
    if not torch.cuda.is_available():
        raise SystemExit("continuous_bench.py measures on the GPU; no CUDA device here")
    dev = torch.device("cuda:0")
    lib = _native.load()
    torch.manual_seed(0)
    from bench import decoder_dims
    dec = genvox_b200.Decoder(**decoder_dims()).to(dev).eval()
    memory, tokens, caps = workload(dev)
    perm = torch.randperm(U_ALL, generator=torch.Generator().manual_seed(13))
    info = device_line()
    print(json.dumps(info), flush=True)

    def batches(mem, ln, cp):
        """bench.py's static batches: 64 utterances each, padded to the batch's longest (made before the timed region)"""
        out = []
        for b0 in range(0, mem.shape[0], BATCH):
            n = int(ln[b0:b0 + BATCH].max())
            out.append((mem[b0:b0 + BATCH, :n].contiguous(), ln[b0:b0 + BATCH], int(cp[b0:b0 + BATCH].max()),
                        int(cp[b0:b0 + BATCH].sum())))
        return out

    def static_arm(bs):
        frames = steps = 0
        for mem, ln, s, f in bs:
            dec.inference(mem, memory_lengths=ln, ignore_gate=True, max_decoder_steps=s)
            frames += f
            steps += s
        return frames, steps

    def continuous_arm(mem, ln, cp):
        dec.inference_continuous(mem, ln, slots=BATCH, max_decoder_steps=MAX_STEPS, frame_caps=cp, ignore_gate=True)
        frames = int(dec.last_n_frames.sum())
        assert frames == int(cp.sum())
        return frames, dec.last_steps_run

    results = []
    for precision in ("fp32", "bf16"):
        dec.precision = precision
        for U in (SHARD, U_ALL):
            for order in ("sorted", "arrival"):
                idx = torch.arange(U) if order == "sorted" else perm[perm < U]
                mem, ln, cp = memory[idx.to(dev)].contiguous(), tokens[idx.to(dev)].contiguous(), caps[idx].contiguous()
                ps, pc = predicted_steps(cp)
                cp_dev = cp.to(dev)
                bs = batches(mem, ln, cp)
                arms = {"static": lambda: static_arm(bs), "continuous": lambda: continuous_arm(mem, ln, cp_dev)}
                static_arm(bs[:1])                                          # warm-up of both arms
                continuous_arm(mem[:2 * BATCH], ln[:2 * BATCH], cp_dev[:2 * BATCH])
                torch.cuda.synchronize()
                times = {k: [] for k in arms}
                for _ in range(args.reps):
                    for name, fn in arms.items():
                        torch.cuda.synchronize()
                        c0 = lib.gvx_launch_count()
                        t0 = time.perf_counter()
                        frames, steps = fn()
                        torch.cuda.synchronize()
                        dt = time.perf_counter() - t0
                        times[name].append((dt, frames, steps, lib.gvx_launch_count() - c0))
                genvox_b200.check_device_errors()
                for name, runs in times.items():
                    best = min(runs)
                    dt, frames, steps, launches = best
                    row = {"precision": precision, "utterances": U, "order": order, "arm": name,
                           "utterances_per_s": U / dt, "seconds": dt, "seconds_all_reps": [round(r[0], 4) for r in runs],
                           "decoder_steps": steps, "predicted_steps": ps if name == "static" else pc,
                           "mel_frames_per_s": frames / dt, "slot_occupancy": frames / (BATCH * steps),
                           "launches_per_step": launches / steps}
                    results.append(row)
                    print(json.dumps(row), flush=True)
    print(f"\n{info['device']}, power limit / max SM clock: {info['power_limit_and_max_sm_clock']}")
    print(f"{'prec':5} {'U':>5} {'order':8} {'arm':11} {'utt/s':>8} {'steps':>7} {'frames/s':>10} {'occup':>6} {'launch/step':>11}")
    for r in results:
        print(f"{r['precision']:5} {r['utterances']:5d} {r['order']:8} {r['arm']:11} {r['utterances_per_s']:8.1f} {r['decoder_steps']:7d} "
              f"{r['mel_frames_per_s']:10.0f} {r['slot_occupancy']:6.3f} {r['launches_per_step']:11.2f}")
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"device": info, "results": results}, fh, indent=1)


if __name__ == "__main__":
    main()
