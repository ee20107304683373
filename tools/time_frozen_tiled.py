"""Times eval-mode autograd (forward + backward with x.requires_grad) with and without SRResNet.grad_budget_bytes on the
GPU: 1 x 1080p whole frame against budgets of 24, 12 and 8 GiB, and 1 x 3840x2160 at 24 and 12 GiB (its whole-frame
frozen workspace, 169 GB, is not run).  Each variant has its own module (trained-like BatchNorm state, default 16 blocks,
x4) so its engines stay warm; variants of one input size are alternated round by round, and the median per variant is
reported with its peak memory, the card's name, power limit and SM clock read in the same run.

    python tools/time_frozen_tiled.py [--rounds 5] [--json out.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def smi(fields):
    r = subprocess.run(["nvidia-smi", f"--query-gpu={fields}", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    import srgan_b200 as S
    from oracle import srgan_oracle as O
    import bn_affine_state as B
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    sd = B.bn_affine_state(O.init_srresnet_state(41), 41)
    cases = [((1, 3, 1080, 1920), [None, 24, 12, 8]), ((1, 3, 2160, 3840), [24, 12])]
    out = {"gpu": smi("name,power.limit,clocks.max.sm"), "rows": []}
    for shape, budgets in cases:
        gen = torch.Generator().manual_seed(42)
        x = torch.rand(*shape, generator=gen).cuda()
        dsr = (torch.randn(shape[0], 3, shape[2] * 4, shape[3] * 4, generator=gen) * 1e-3).cuda()
        mods = {}
        for b in budgets:
            g = S.SRResNet()
            g.load_state_dict(sd)
            g = g.cuda().eval()
            g.grad_budget_bytes = None if b is None else b << 30
            mods[b] = g
        times = {b: [] for b in budgets}
        peaks = {b: 0 for b in budgets}
        clocks = []

        def step(b):
            g = mods[b]
            xx = x.clone().requires_grad_()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            s0.record()
            g(xx).backward(dsr)
            s1.record()
            torch.cuda.synchronize()
            for p in g.parameters():
                p.grad = None
            return s0.elapsed_time(s1), torch.cuda.max_memory_allocated() - base

        for b in budgets:
            step(b)                                       # warm-up: engines, workspaces, plans
        for r in range(a.rounds):
            for b in (budgets if r % 2 == 0 else budgets[::-1]):
                ms, peak = step(b)
                times[b].append(ms)
                peaks[b] = max(peaks[b], peak)
            clocks.append(smi("clocks.sm"))
        for b in budgets:
            g = mods[b]
            row = {"input": "x".join(map(str, shape)), "budget_gib": b, "median_ms": statistics.median(times[b]),
                   "min_ms": min(times[b]), "step_peak_rise_gib": peaks[b] / 2**30,
                   "engine_workspace_gib": g.last_engine().ws.numel() / 2**30}
            if b is not None:
                win_h, win_w, n, tiles = g._frozen_tiles_plan(shape[0], shape[2], shape[3], x.device)
                row.update(windows=len(tiles), window=f"{win_h}x{win_w}", per_call=n,
                           recompute=len(tiles) * win_h * win_w / (shape[0] * shape[2] * shape[3]))
            out["rows"].append(row)
            print(json.dumps(row))
        out.setdefault("sm_clock_samples", []).extend(clocks)
        del mods
        torch.cuda.empty_cache()
    print("gpu (name, power limit, max SM clock):", out["gpu"])
    print("SM clock samples:", out["sm_clock_samples"])
    if a.json:
        with open(a.json, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
