"""Developer tool (GPU box): throughput and peak memory of the spatially tiled eval forward (SRResNet.tile_budget_bytes).

    python tools/time_tiled.py [--reps 5] [--out DIR]

Default SRResNet (16 residual blocks, x4), eval mode, no_grad.  For 8 x 3 x 1080 x 1920 LR frames it runs budget None
(the frame streaming path: one frame per engine call, ~7.4 GB of workspace) and tile budgets of 4, 2 and 1 GB.  Each
budget gets a fresh module (same seeded weights, no engine yet): one cold call, then `--reps` timed calls (CUDA events
around the whole forward; the median is reported as frames/s).  Per budget it reports the window plan (window size,
windows per frame, window pixels / frame pixels), the engine workspace the module holds afterwards, and
torch.cuda.max_memory_allocated over what was allocated before the cold call (engine workspace + output + transients).  Then one 3840 x 2160 and one 7680 x 4320 LR
frame at a 6 GB tile budget.  Every tiled output is compared bitwise with the budget-None output of the same input
(skipped for the 8K frame, whose whole-frame workspace is ~119 GB).  The card name, power limit and max SM clock are read
in the same run (read-only nvidia-smi query), and the SM clock is sampled during the timed 1080p calls, as bench.py does."""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import srgan_b200 as S                       # noqa: E402


def sm_clocks():
    r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=clocks.sm,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True)
    try:
        cur, mx = (int(v) for v in r.stdout.strip().split(","))
        return cur, mx
    except ValueError:
        return None, None


def fresh_generator():
    """the same seeded weights every time, on a module with no engine yet"""
    torch.manual_seed(0)
    return S.SRResNet().cuda().eval()


def pool_workspace_bytes(g):
    return sum(e.ws.numel() for pool in g._rt["engines"].values() for e in pool if e.ws is not None)


def run(x, budget, reps):
    """fresh module: the first (cold) call plans, creates and binds its engine, so the peak memory measured from before it
    includes the engine workspace the budget governs, plus the output"""
    g = fresh_generator()
    g.tile_budget_bytes = budget
    torch.cuda.synchronize()
    gc.collect()                              # the previous budget's module and engines
    torch.cuda.empty_cache()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    with torch.no_grad():
        out = g(x)                            # cold call: plan, engine, module loads (not timed)
        torch.cuda.synchronize()
        times, clocks = [], []
        for _ in range(reps):
            out = None
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = g(x)
            b.record()
            clocks.append(sm_clocks()[0])
            torch.cuda.synchronize()
            times.append(a.elapsed_time(b))
        peak = torch.cuda.max_memory_allocated() - before
    ms = statistics.median(times)
    res = {"budget_gb": None if budget is None else budget / 2 ** 30, "ms": round(ms, 2),
           "frames_per_s": round(x.shape[0] / ms * 1e3, 3), "peak_rise_gb": round(peak / 2 ** 30, 3),
           "output_gb": round(out.numel() * 4 / 2 ** 30, 3), "engine_workspace_gb": round(pool_workspace_bytes(g) / 2 ** 30, 3),
           "engine_N": g.last_engine().N, "sm_mhz_samples": [c for c in clocks if c is not None]}
    key = ("tiles", x.shape[0], x.shape[2], x.shape[3], budget)
    if budget is not None and key in g._rt:
        wh, ww, per_call, tiles = g._rt[key]
        per_frame = len(tiles) // x.shape[0]
        res.update({"window": [wh, ww], "windows_per_frame": per_frame, "windows_per_call": per_call,
                    "pixel_ratio": round(per_frame * wh * ww / (x.shape[2] * x.shape[3]), 4)})
    return g, out, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_tiled.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[torch.cuda.current_device()] if card else 'unknown'}", flush=True)
    results = []
    x = torch.rand(8, 3, 1080, 1920, device="cuda")
    ref = None
    for budget in (None, 4 << 30, 2 << 30, 1 << 30):
        g, out, res = run(x, budget, args.reps)
        if budget is None:
            ref = out.clone()
        else:
            res["bitwise_equal_to_untiled"] = bool(torch.equal(out, ref))
        del out, g
        results.append(dict(res, frames="8x1080x1920"))
        print(json.dumps(results[-1]), flush=True)
    del ref
    for (h, w) in ((2160, 3840), (4320, 7680)):
        x = torch.rand(1, 3, h, w, device="cuda")
        t0 = time.time()
        g, out, res = run(x, 6 << 30, 1)
        res["wall_s_incl_cold_call"] = round(time.time() - t0, 2)
        if h == 2160:
            g.tile_budget_bytes = None
            with torch.no_grad():
                res["bitwise_equal_to_untiled"] = bool(torch.equal(out, g(x)))
        del out, g
        results.append(dict(res, frames=f"1x{h}x{w}"))
        print(json.dumps(results[-1]), flush=True)
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_tiled.json"), "w") as f:
            json.dump({"card": card, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
