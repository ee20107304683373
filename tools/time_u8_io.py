"""Developer tool (GPU box): time and peak memory of the 8-bit eval path (SRResNet.upscale_u8) against the fp32 path.

    python tools/time_u8_io.py [--reps 5] [--out DIR]

Default SRResNet (16 residual blocks, x4), eval mode, seeded weights, random uint8 frames.  Three ways to upscale the
same uint8 N x H x W x 3 frames, alternated call by call in one process (a, b, c, a, b, c, ...):

  (a) transformers.to_tensor + the fp32 forward (fp32 NCHW SR out);
  (b) (a) + the torch quantise / permute: (sr.clamp(0, 1) * 255).round().to(uint8).permute(0, 2, 3, 1).contiguous();
  (c) upscale_u8 (uint8 NHWC SR out).

Each call is timed with CUDA events around the whole call (median of --reps after one untimed warm-up call per way);
its peak is torch.cuda.max_memory_allocated over what was allocated before the call, so it counts the output and every
temporary but not the input frames or the engines, which are created by the warm-up call.  Workloads: 8 x 1080 x 1920 with
the default stream budget (frame streaming, one frame per engine call), and one 7680 x 4320 frame at a 4 GiB tile budget
(spatial windows).  (b) and (c) are compared bitwise.  The card name, power limit and max SM clock are read in the same
run (read-only nvidia-smi query)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import srgan_b200 as S                       # noqa: E402


def way_a(g, frames):
    return g(S.transformers.to_tensor(frames))


def way_b(g, frames):
    return (way_a(g, frames).clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def way_c(g, frames):
    return g.upscale_u8(frames)


WAYS = {"a_to_tensor_fp32_forward": way_a, "b_a_plus_torch_quantise": way_b, "c_upscale_u8": way_c}


def one_call(fn, g, frames):
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn(g, frames)
    b.record()
    torch.cuda.synchronize()
    return out, a.elapsed_time(b), torch.cuda.max_memory_allocated() - before


def workload(name, frames, tile_budget, reps):
    torch.manual_seed(0)
    g = S.SRResNet().cuda().eval()
    g.tile_budget_bytes = tile_budget
    times = {k: [] for k in WAYS}
    peaks = {k: 0 for k in WAYS}
    with torch.no_grad():
        for k, fn in WAYS.items():                        # warm-up: plans, engines, module loads
            one_call(fn, g, frames)
        ref = out_c = None
        for _ in range(reps):
            for k, fn in WAYS.items():
                out, ms, peak = one_call(fn, g, frames)
                times[k].append(ms)
                peaks[k] = max(peaks[k], peak)
                if k == "b_a_plus_torch_quantise":
                    ref = out
                elif k == "c_upscale_u8":
                    out_c = out
                del out
        equal = bool(torch.equal(ref, out_c))
    res = {"workload": name, "tile_budget_gib": None if tile_budget is None else tile_budget / 2 ** 30, "reps": reps,
           "bitwise_b_equals_c": equal}
    for k in WAYS:
        res[k] = {"median_ms": round(statistics.median(times[k]), 2), "min_ms": round(min(times[k]), 2),
                  "peak_rise_gib": round(peaks[k] / 2 ** 30, 3)}
    del g, ref, out_c
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_u8_io.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    card = card[torch.cuda.current_device()] if card else "unknown"
    print(f"card: {card}", flush=True)
    gen = torch.Generator(device="cuda").manual_seed(1)
    results = []
    frames = torch.randint(0, 256, (8, 1080, 1920, 3), dtype=torch.uint8, device="cuda", generator=gen)
    results.append(workload("8x1080x1920", frames, None, args.reps))
    print(json.dumps(results[-1]), flush=True)
    del frames
    frames = torch.randint(0, 256, (1, 4320, 7680, 3), dtype=torch.uint8, device="cuda", generator=gen)
    results.append(workload("1x4320x7680", frames, 4 << 30, max(1, args.reps // 2)))
    print(json.dumps(results[-1]), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_u8_io.json"), "w") as f:
            json.dump({"card": card, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
