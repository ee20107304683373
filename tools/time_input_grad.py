"""Developer tool (GPU box): what an input gradient through SRResNet costs at the cfg2 geometry (16 x 3 x 96 x 96, default
SRResNet: 16 residual blocks, x4).

    python tools/time_input_grad.py [--calls 200] [--n 16 --h 96 --w 96]

Four variants, alternated call by call in one run so that they see the same clocks and neighbours:
  train       train-mode forward + backward, x does not require grad (every parameter gradient)
  train+dx    the same with x.requires_grad: adds conv1's filter pack and data gradient
  input-only  train mode, every parameter frozen, x.requires_grad: the data-gradient chain only
  frozen      eval mode, x.requires_grad: running BatchNorm statistics, x.grad plus every parameter gradient
CUDA events around the forward and around the backward of every call, after every shape was warmed up; medians over
`--calls` calls per variant.  Prints the card name, power limit and max SM clock read in the same run (nvidia-smi,
read-only query) and the algorithmic GFLOP of conv1's data gradient, computed from the shapes."""
import argparse
import copy
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import srgan_b200 as S                       # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--n", type=int, default=16)
    ap.add_argument("--h", type=int, default=96)
    ap.add_argument("--w", type=int, default=96)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_input_grad.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[torch.cuda.current_device()] if card else 'unknown'}")
    N, H, W = args.n, args.h, args.w
    torch.manual_seed(0)
    g = S.SRResNet().cuda()
    g_only = copy.deepcopy(g).requires_grad_(False)
    gen = torch.Generator(device="cuda").manual_seed(1)
    lr = torch.rand(N, 3, H, W, device="cuda", generator=gen)
    dsr = torch.randn(N, 3, 4 * H, 4 * W, device="cuda", generator=gen) * 1e-4

    def run(name):
        mod = g_only if name == "input-only" else g
        mod.train(name != "frozen")
        x = lr.requires_grad_(False) if name == "train" else lr.detach().requires_grad_()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        y = mod(x)
        e1.record()
        y.backward(dsr)
        e2.record()
        return e0, e1, e2

    names = ["train", "train+dx", "input-only", "frozen"]
    for _ in range(args.warmup):
        for n in names:
            run(n)
            g.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    ev = {n: [] for n in names}
    for _ in range(args.calls):
        for n in names:
            ev[n].append(run(n))
            g.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    med = {}
    for n in names:
        fwd = statistics.median(a.elapsed_time(b) for a, b, _ in ev[n])
        bwd = statistics.median(b.elapsed_time(c) for _, b, c in ev[n])
        tot = statistics.median(a.elapsed_time(c) for a, _, c in ev[n])
        med[n] = (fwd, bwd, tot)
        print(f"{n:>10}: forward {fwd:.3f} ms, backward {bwd:.3f} ms, forward + backward {tot:.3f} ms "
              f"(medians over {args.calls} calls)")
    gflop = 2.0 * 64 * 3 * 81 * N * H * W / 1e9
    d = med["train+dx"][2] - med["train"][2]
    print(f"conv1 data gradient: {gflop:.2f} GFLOP algorithmic; train+dx - train = {d * 1e3:.0f} us (pack + conv)"
          + (f" -> {gflop / (d * 1e-3) / 1e3:.1f} TFLOP/s" if d > 0 else ""))
    print(f"backward: full (train+dx) {med['train+dx'][1]:.3f} ms vs input-only {med['input-only'][1]:.3f} ms "
          f"({100 * (1 - med['input-only'][1] / med['train+dx'][1]):.0f}% less)")
    print(f"forward + backward: frozen {med['frozen'][2]:.3f} ms vs train {med['train+dx'][2]:.3f} ms "
          f"(ratio {med['frozen'][2] / med['train+dx'][2]:.3f})")


if __name__ == "__main__":
    main()
