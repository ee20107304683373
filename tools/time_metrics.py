"""Developer tool (GPU box): time srg_image_metrics (per-image PSNR + SSIM, evaluation.image_metrics) at the reference's
validation geometry, 12 x 3 x 512 x 1024 fp32, against the HBM roofline, next to the fp64 CPU oracle's time for one batch.

    python tools/time_metrics.py [--calls 400] [--pairs 4] [--n 12 --h 512 --w 1024]

CUDA events around every call; the inputs rotate through `--pairs` distinct SR / HR pairs (4 pairs of 151 MB = 604 MB, far
beyond the 126 MB L2), so each call reads its 8 bytes per element from HBM.  Prints the card name, power limit and max SM
clock read in the same run (nvidia-smi, read-only query)."""
import argparse
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import srgan_b200 as S                       # noqa: E402
from oracle import srgan_oracle as O         # noqa: E402
import ssim_oracle                           # noqa: E402  (tests/ssim_oracle.py)

HBM_GBS = 6549.4                             # the project's HBM figure (DESIGN section 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=400)
    ap.add_argument("--pairs", type=int, default=4)
    ap.add_argument("--n", type=int, default=12)
    ap.add_argument("--h", type=int, default=512)
    ap.add_argument("--w", type=int, default=1024)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_metrics.py needs a CUDA device")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[torch.cuda.current_device()] if card else 'unknown'}")
    N, H, W = args.n, args.h, args.w
    g = torch.Generator(device="cuda").manual_seed(0)
    pairs = []
    for _ in range(args.pairs):
        hr = torch.rand(N, 3, H, W, device="cuda", generator=g)
        pairs.append(((hr + 0.03 * torch.randn(N, 3, H, W, device="cuda", generator=g)).clamp_(0, 1), hr))
    for sr, hr in pairs:                      # warm-up: module load, scratch allocation
        S.image_metrics(sr, hr)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.calls)]
    for i, (e0, e1) in enumerate(ev):
        sr, hr = pairs[i % len(pairs)]
        e0.record()
        S.image_metrics(sr, hr)
        e1.record()
    torch.cuda.synchronize()
    us = sorted(1e3 * e0.elapsed_time(e1) for e0, e1 in ev)
    med = statistics.median(us)
    nbytes = 8.0 * N * 3 * H * W
    gbs = nbytes / (med * 1e-6) / 1e9
    print(f"srg_image_metrics {N}x3x{H}x{W}: median {med:.1f} us per call over {args.calls} calls "
          f"(p10 {us[len(us) // 10]:.1f}, p90 {us[9 * len(us) // 10]:.1f}); {nbytes / 1e6:.1f} MB read -> {gbs:.1f} GB/s "
          f"algorithmic = {100 * gbs / HBM_GBS:.1f}% of {HBM_GBS} GB/s")
    sr, hr = (t.cpu() for t in pairs[0])
    t0 = time.perf_counter()
    ref = [(O.psnr(sr[n], hr[n]), ssim_oracle.ssim(sr[n], hr[n])) for n in range(N)]
    t_cpu = time.perf_counter() - t0
    psnr, ssim = S.image_metrics(*pairs[0])
    dp = max(abs(float(psnr[n]) - ref[n][0]) for n in range(N))
    ds = max(abs(float(ssim[n]) - ref[n][1]) for n in range(N))
    print(f"fp64 CPU oracle (torch, {torch.get_num_threads()} threads): {t_cpu:.2f} s for the batch; "
          f"max |device - oracle|: PSNR {dp:.2e} dB, SSIM {ds:.2e}")


if __name__ == "__main__":
    main()
