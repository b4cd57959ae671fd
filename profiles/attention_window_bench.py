"""Cost of the attention constraint (Decoder.attention_window) per decoder step, on one GPU.

The constraint adds one N-wide (value, index) block reduction per row and step to the forward attention kernel, and only
when a window is set; this measures what that costs in whole decoder steps.

  static      BASELINE configs[1]'s shape: Decoder.inference on 64 rows of 150 tokens, 1000 fixed steps (gate ignored);
  continuous  Decoder.inference_continuous with 64 slots on 256 utterances of 75-150 tokens, each stopped at a frame cap
              of tokens x U[4.5, 7.5] (seeded, at most 1000; random-init weights make no realistic gate stops), so both
              arms run the same decoder steps.

Each runs unconstrained and with the window (1, 3) (ESPnet's defaults), alternating in one process, `--reps` times; the
best time of each arm gives ms per decoder step.  The device name and power limit are read in the same run.
Usage: python profiles/attention_window_bench.py [--reps 3] [--precision fp32] [--out FILE.json]
"""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from continuous_bench import device_line  # noqa: E402

B, N, STEPS = 64, 150, 1000          # BASELINE configs[1]
U_CONT = 256
WINDOWS = {"unconstrained": None, "window_1_3": (1, 3)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--precision", default="fp32", choices=["fp32", "bf16"])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attention_window_bench.py measures on the GPU; no CUDA device here")
    import genvox_b200
    from bench import decoder_dims
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    dec = genvox_b200.Decoder(**decoder_dims()).to(dev).eval()
    dec.precision = args.precision
    info = device_line()
    print(json.dumps(info), flush=True)

    memory = (0.5 * torch.randn(B, N, 512, generator=torch.Generator().manual_seed(1))).to(dev)
    g = torch.Generator().manual_seed(7)
    tokens = torch.randint(75, N + 1, (U_CONT,), generator=g)
    cmem = 0.5 * torch.randn(U_CONT, N, 512, generator=torch.Generator().manual_seed(2))
    for u, n in enumerate(tokens.tolist()):
        cmem[u, n:] = 0
    rate = 4.5 + 3.0 * torch.rand(U_CONT, generator=torch.Generator().manual_seed(11))
    caps = torch.clamp((tokens.double() * rate.double()).floor().long(), 1, STEPS).to(torch.int32).to(dev)
    cmem, tokens = cmem.to(dev), tokens.to(dev)

    def static(win):
        dec.inference(memory, ignore_gate=True, max_decoder_steps=STEPS, attention_window=win)
        return STEPS

    def continuous(win):
        dec.inference_continuous(cmem, tokens, slots=64, max_decoder_steps=STEPS, frame_caps=caps, ignore_gate=True,
                                 return_alignments=False, attention_window=win)
        return dec.last_steps_run

    for win in WINDOWS.values():                       # warm-up: weight packing, kernel attributes, both arms
        dec.inference(memory, ignore_gate=True, max_decoder_steps=8, attention_window=win)
        dec.inference_continuous(cmem[:8], tokens[:8], slots=64, max_decoder_steps=8, ignore_gate=True, attention_window=win)
    torch.cuda.synchronize()

    results = []
    for arm_name, fn in (("static", static), ("continuous", continuous)):
        runs = {k: [] for k in WINDOWS}
        for _ in range(args.reps):
            for name, win in WINDOWS.items():
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                steps = fn(win)
                torch.cuda.synchronize()
                runs[name].append(((time.perf_counter() - t0) * 1e3 / steps, steps))
        genvox_b200.check_device_errors()
        best = {k: min(v) for k, v in runs.items()}
        row = {"arm": arm_name, "precision": args.precision, "decoder_steps": best["unconstrained"][1],
               **{f"ms_per_step_{k}": round(v[0], 4) for k, v in best.items()},
               **{f"ms_per_step_{k}_all_reps": [round(r[0], 4) for r in v] for k, v in runs.items()},
               "window_cost_ms_per_step": round(best["window_1_3"][0] - best["unconstrained"][0], 4),
               "window_cost_percent": round(100.0 * (best["window_1_3"][0] / best["unconstrained"][0] - 1.0), 2)}
        assert best["window_1_3"][1] == best["unconstrained"][1]
        results.append(row)
        print(json.dumps(row), flush=True)
    print(f"\n{info['device']}, power limit / max SM clock: {info['power_limit_and_max_sm_clock']}")
    for r in results:
        print(f"{r['arm']:11} {r['precision']}: {r['ms_per_step_unconstrained']:.4f} ms/step unconstrained, "
              f"{r['ms_per_step_window_1_3']:.4f} with (1, 3): {r['window_cost_ms_per_step']:+.4f} ms ({r['window_cost_percent']:+.2f} %)")
    if args.out:
        with open(args.out, "w") as fh:
            json.dump({"device": info, "results": results}, fh, indent=1)


if __name__ == "__main__":
    main()
