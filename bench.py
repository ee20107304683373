#!/usr/bin/env python
"""Benchmark of the SR-GAN train step (BASELINE.json metric: train LR-patches/sec; conv tensor-pipe roofline).

    python bench.py --gpus 1 --steps 20 --warmup 3                 # this repo's CUDA path on cuda:0
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU: BASELINE configs[2], global batch 256
    python bench.py --impl reference --steps 3 --warmup 1           # the UNMODIFIED reference step on the host cores
    python bench.py --gpus 1 --steps 20 --warmup 3 --dump-outputs out/  # also write the last timed step's outputs

--dump-outputs DIR writes, right after the timed steps, what a caller of the timed path holds after its last step:
losses.npy (the [K, 4] loss rows MultiGeneratorGAN.step returned) and generator<i>_state.npy (discriminator_state.npy
at gan-native), every floating-point state_dict entry of that model after the update, flattened in state_dict order;
infer-1080p writes sr.npy, a fixed sample of the upscaled frames.  On N > 1 GPUs rank 0 writes them.  Inputs and initial
weights are seeded, so two builds run with the same arguments can be compared output for output.

Workload (N=1): BASELINE.json configs[1] -- K=3 generators (count inferred from src/main.py:28), each doing the
reference's train_generator step (SRResNet fwd+bwd, ReconstructionLoss, Adam) on one batch of 16x3x96x96 synthetic LR
patches (HR 16x3x384x384), bf16 operands / fp32 accumulate.  The reference Discriminator raises on 384x384 HR inputs
(SURVEY Appendix E), so like the reference's HEAD the discriminator step is not part of this configuration.
One step = all K generator updates on one batch; value = batch patches / step time, summed over ranks.

Workload (N > 1): BASELINE.json configs[2] -- the same step batch-sharded over N GPUs at GLOBAL batch 256 (256/N patches
per GPU), NCCL gradient all-reduce + SyncBatchNorm; the line also carries the weak-scaling figure at 16 patches per GPU
("weak16") so that both readings of the scaling question are on record.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "srgan_train_lr_patches_per_sec"
UNIT = "patches/s"
FLOP_PER_LR_PIXEL_FWD_BWD = 13277952.0          # SURVEY Appendix A: generator fwd+bwd, conv MACs x 2
TRUNK_CONV_FLOP_PER_PIXEL = 2.0 * 64 * 64 * 9   # one 3x3 64->64 conv (fprop or dgrad) per LR pixel


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--generators", type=int, default=3)
    ap.add_argument("--batch", type=int, default=None, help="LR patches per GPU per step (default: 16 on one GPU = "
                    "configs[1]; 256 / N on N > 1 GPUs = configs[2])")
    ap.add_argument("--no-weak16", action="store_true", help="N > 1: skip the secondary 16-patches-per-GPU measurement")
    ap.add_argument("--no-hbm", action="store_true", help="skip the HBM roofline leg (memory-bound kernels timed alone)")
    ap.add_argument("--lr-size", type=int, default=96)
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "gan-native", "infer-1080p"],
                    help="cfg2: BASELINE configs[1] (default).  gan-native: D update + all generators in GAN mode at the "
                         "reference's native geometry (LR 128x256, batch 12), where its Discriminator is valid")
    ap.add_argument("--ref-sample-batch", type=int, default=4, help="patches per step of the CPU reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-sync-each-step", action="store_true", help="e2e leg: wait for every step's losses before "
                    "enqueuing the next step (default: read them one step late)")
    ap.add_argument("--syncbn", default="peer", choices=["peer", "nccl", "none"], help="SyncBatchNorm transport for N > 1: fused "
                    "NVLink peer-memory exchange kernel (default) or ncclAllReduce between reduce and finalize kernels")
    ap.add_argument("--no-stream", action="store_true", help="infer-1080p: one engine call for the whole batch instead of "
                    "streaming chunks of frames (A/B; materialises every frame's activations)")
    ap.add_argument("--no-graphs", action="store_true", help="enqueue every kernel from the host instead of replaying "
                    "one captured CUDA graph per generator step")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last "
                    "timed step returned and the model state it left as DIR/<name>.npy (float32, at most 64 MB in all), "
                    "so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's CUDA path (--impl ours)")
    return a


def geometry(a):
    if a.workload == "gan-native":
        return (a.batch or 12), 128, 256     # batch 12 (src/train.py:94), LR 128x256 (src/transformers.py:74)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.batch is None:
        return (16 if world == 1 else max(256 // world, 1)), a.lr_size, a.lr_size
    return a.batch, a.lr_size, a.lr_size


def workload_name(a):
    b, h, w = geometry(a)
    if a.workload == "gan-native":
        return (f"gan-native: train_discriminator + {a.generators} generators x train_generator in GAN mode "
                f"(SRResNet fwd+bwd, ReconstructionLoss + tanh adversarial term through D, Adam), {b}x3x{h}x{w} LR -> x4 HR per GPU")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cfg = "cfg2" if world == 1 else f"cfg3 (global batch {b * world} over {world} GPUs)"
    return (f"{cfg}: {a.generators} generators x train_generator (SRResNet fwd+bwd + ReconstructionLoss + Adam), "
            f"{b}x3x{h}x{w} LR -> x4 HR per GPU, pixel-loss mode (reference D invalid at this HR size)")


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Writes every tensor of ``arrays`` as ``path/<name>.npy`` in float32, 64 MB in all at most.  Tensors are taken
    smallest first and each may use an equal part of the budget still left; one larger than its part is written as
    the flat elements at a fixed set of indices (numpy default_rng(0), sorted, duplicates dropped), so that runs with
    the same arguments write the same elements."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    left = DUMP_BUDGET_BYTES - 1024 * len(arrays)         # room for the .npy headers
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel())):
        t = t.detach().float()
        share = left // (len(arrays) - i) // 4
        if t.numel() > share:
            idx = np.unique(np.random.default_rng(0).integers(0, t.numel(), share))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        left -= 4 * t.numel()
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy())


def state_vector(module):
    """Every floating-point entry of ``module.state_dict()`` (parameters and BatchNorm running statistics), flattened
    and concatenated in state_dict order."""
    import torch
    return torch.cat([v.detach().reshape(-1).float() for v in module.state_dict().values() if v.is_floating_point()])


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=self.f,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.f.close()
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
            sm = sorted(float(r[0]) for r in rows if r[0].replace(".", "").isdigit())
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][1])
                out["power_w_max"] = max(float(r[2]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for i, nme in enumerate(names):
                if any(len(r) > 4 + i and r[4 + i].strip().lower() == "active" for r in rows):
                    out["reasons"].append(nme)
            out["samples"] = len(rows)
        except Exception:
            pass
        return out


# ----------------------------------------------------------------------------------------------------------------
# CPU arithmetic of the reference (oracle port): used by --impl reference and by the cpu_baseline leg only
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(a, steps, warmup, budget_s=150.0):
    """K x train_generator on the host cores, on a bounded sample of the batch.  Runs the UNMODIFIED reference
    (src/train.py:175-203 with src/models.py / src/utils.py, copied verbatim into the git-ignored oracle/_ref by
    oracle/make_ref.py) when that copy travelled with the snapshot -> kind "reference"; otherwise the oracle's
    restatement of the same arithmetic -> kind "port".  Returns (patches/s, s/step, cores, sample text, kind, batch)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    size = a.lr_size
    kind = "port"
    try:
        from oracle import make_ref
        if make_ref.available():
            models, train, utils = make_ref.import_reference()
            kind = "reference"
    except Exception:
        kind = "port"
    if kind == "reference":
        def build():
            torch.manual_seed(0)
            gens = []
            for s_ in range(a.generators):
                torch.manual_seed(s_)
                gens.append(models.SRResNet())
            opts = [torch.optim.Adam(g.parameters(), lr=1e-4) for g in gens]
            crit = utils.ReconstructionLoss()
            torch.manual_seed(100)
            disc = models.Discriminator()          # passed like the reference's loop does; unused at HEAD (g_d_loss = 0)

            def step(lr, hr):
                for g, o in zip(gens, opts):
                    train.train_generator(g, disc, lr, hr, None, crit, o)
            return step
        what = "UNMODIFIED reference src/train.py:train_generator (anomaly detection on, as upstream)"
    else:
        from oracle import srgan_oracle as O

        def build():
            gens = [O.init_srresnet_state(s_) for s_ in range(a.generators)]
            opts = [O.AdamState([sd[k] for k in O.trainable_keys(sd)], lr=1e-4) for sd in gens]

            def step(lr, hr):
                for sd, opt in zip(gens, opts):
                    O.train_generator_step(sd, opt, lr, hr)
            return step
        what = "oracle restatement of the reference step (oracle/srgan_oracle.py; oracle/_ref not present)"
    # bounded sample: calibrate on one patch, then the largest sample batch (<= --ref-sample-batch) inside the budget
    step = build()
    t0 = time.perf_counter()
    step(torch.rand(1, 3, size, size), torch.rand(1, 3, 4 * size, 4 * size))
    t_one = time.perf_counter() - t0
    b = max(1, min(a.ref_sample_batch, int(budget_s / max((steps + warmup) * t_one, 1e-9))))
    step = build()
    torch.manual_seed(0)
    lr = torch.rand(b, 3, size, size)
    hr = torch.rand(b, 3, 4 * size, 4 * size)
    for _ in range(warmup):
        step(lr, hr)
    t0 = time.perf_counter()
    for _ in range(steps):
        step(lr, hr)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    try:
        torch.autograd.set_detect_anomaly(False)
    except Exception:
        pass
    sample = (f"{a.generators} generators x {what} on {b}x3x{size}x{size} LR patches per step (a bounded sample of the "
              f"16-patch cfg2 batch: patches/s = {b} / step time), fp32, torch CPU kernels, {cores} threads")
    return b / dt, dt, cores, sample, kind, b


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    val, dt, cores, sample, kind, b = cpu_reference_steps(a, a.steps, a.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": ("strong" if (int(os.environ.get("WORLD_SIZE", "1")) > 1 and a.batch is None and a.workload == "cfg2") else "weak"),
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the same workload keys as the GPU arm prints (the arm times a bounded sample of that workload: cpu_baseline.sample)
        "config": {"workload": workload_name(a), "generators": a.generators, "batch_per_gpu": geometry(a)[0],
                   "global_batch": geometry(a)[0] * int(os.environ.get("WORLD_SIZE", "1")),
                   "lr_hw": [geometry(a)[1], geometry(a)[2]], "upscale": 4,
                   "parallelism": f"dp{int(os.environ.get('WORLD_SIZE', '1'))}", "sample_batch": b,
                   "note": ("the unmodified reference sources run from oracle/_ref (copied verbatim by oracle/make_ref.py, "
                            "git-ignored)" if kind == "reference" else
                            "oracle/_ref did not travel: reference arithmetic restated on torch CPU kernels (oracle/srgan_oracle.py)")},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
def run_infer(a):
    """BASELINE configs[3]: generator-only inference (eval mode, running BatchNorm statistics) on synthetic 1920x1080 LR
    frames, batch 8 per GPU, x4 upscale -> 7680x4320.  Secondary workload: frames/s, not the headline metric."""
    import torch
    import srgan_b200 as S
    torch.cuda.set_device(0)
    torch.manual_seed(0)
    g = S.SRResNet().cuda().eval()
    if a.no_stream:
        g.stream_budget_bytes = None
    B, H, W = (a.batch or 8), 1080, 1920
    x = torch.rand(B, 3, H, W, device="cuda")
    sampler = ClockSampler(0)
    with torch.no_grad():
        for _ in range(max(a.warmup, 1)):
            y = g(x)
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler.start()
        e0.record()
        for _ in range(a.steps):
            y = g(x)
        e1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"sr": y})
    ms = e0.elapsed_time(e1) / a.steps
    flop = 4436352.0 * H * W * B
    pk, src = peaks()
    frames_per_call = g.last_engine().N
    print(json.dumps({"metric": "srgan_infer_lr_frames_per_sec", "value": B / (ms * 1e-3), "unit": "frames/s", "n_gpus": 1,
                      "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": f"infer-1080p: SRResNet eval forward, {B}x3x{H}x{W} LR -> x4", "out_shape": list(y.shape),
                                 "algorithmic_tflops": flop / (ms * 1e-3) / 1e12,
                                 "frac_of_bf16_sustained_peak": flop / (ms * 1e-3) / 1e12 / float(pk["bf16_tflops_sustained"]),
                                 "frames_per_engine_call": frames_per_call,
                                 "peak_device_memory_gb": torch.cuda.max_memory_allocated() / 1e9},
                      "clocks": clocks, "gpu_launches": int(S.lib().srg_total_launches())}), flush=True)


def hbm_roofline(S, torch, dev, B, LH, LW, pk):
    """Achieved HBM GB/s of the memory-bound kernels of the step, each timed ALONE with CUDA events on cfg-shaped
    tensors through its per-operator C-ABI entry point.  Every launch works on a different one of `nbuf` buffer sets
    (together far larger than the 126 MB L2), so the algorithmic bytes really come from / go to HBM.  The `reps` launches
    are captured into a CUDA graph and the replay is timed (the way the step runs them): host enqueue time per launch
    through ctypes is of the order of these kernels' durations and would otherwise be part of the figure."""
    from ctypes import c_void_p
    L = S.lib()

    def stp():                                            # the CURRENT stream (the capture stream inside torch.cuda.graph)
        return c_void_p(torch.cuda.current_stream().cuda_stream)
    P = B * LH * LW
    act_bytes = P * 128                                     # one [P][64] bf16 tensor
    nbuf = max(4, int(600e6 // (3 * act_bytes)) + 1)
    bufs = [[torch.randn(P, 64, device=dev).to(torch.bfloat16) for _ in range(3)] for _ in range(nbuf)]
    coef = torch.rand(5, 64, device=dev) + 0.5
    rows = L.srg_bn_stats_rows(P)
    partials = torch.empty(rows, 128, device=dev)
    hr = [torch.rand(B, 3, 4 * LH, 4 * LW, device=dev) for _ in range(2)]
    sr = [torch.rand(B, 3, 4 * LH, 4 * LW, device=dev) for _ in range(2)]
    scratch = torch.empty(int(L.srg_recon_loss_scratch_bytes()), dtype=torch.uint8, device=dev)
    e_buf, g_buf, dsr = torch.empty_like(sr[0]), torch.empty_like(sr[0]), torch.empty_like(sr[0])
    losses = torch.empty(2, device=dev)
    img_bytes = hr[0].numel() * 4

    def p(t):
        return c_void_p(t.data_ptr())

    def k_apply_relu(i):
        a_, b_, c_ = bufs[i % nbuf]
        L.srg_bn_apply(p(a_), p(coef[0]), p(coef[1]), None, 1, p(c_), P, stp())

    def k_apply_skip(i):
        a_, b_, c_ = bufs[i % nbuf]
        L.srg_bn_apply(p(a_), p(coef[0]), p(coef[1]), p(b_), 0, p(c_), P, stp())

    def k_stats2(i):
        a_, b_, c_ = bufs[i % nbuf]
        L.srg_bn_stats(p(a_), p(b_), P, p(partials), stp())

    def k_bwd_apply(i):
        a_, b_, c_ = bufs[i % nbuf]
        L.srg_bn_backward_apply(p(a_), p(b_), p(coef[2]), p(coef[3]), p(coef[4]), p(c_), P, stp())

    def k_loss(i):
        h_, s_ = hr[i % 2], sr[i % 2]
        L.srg_recon_loss_forward(p(h_), p(s_), B, 3, 4 * LH, 4 * LW, p(scratch), scratch.numel(), p(e_buf), p(g_buf), p(losses), stp())
        L.srg_recon_loss_backward(p(h_), p(s_), B, 3, 4 * LH, 4 * LW, p(scratch), p(e_buf), p(g_buf), None, None, p(dsr), 1.0, stp())

    cases = [
        ("bn_apply_kernel<relu> (BatchNorm apply + ReLU, src/models.py:23)", k_apply_relu, 2 * act_bytes),
        ("bn_apply_kernel<skip> (BatchNorm apply + residual add, src/models.py:24-25)", k_apply_skip, 3 * act_bytes),
        ("chan_reduce_kernel<two> (BatchNorm backward sums: sum dz, sum dz*y)", k_stats2, 2 * act_bytes),
        ("bn_bwd_apply_kernel (BatchNorm input gradient)", k_bwd_apply, 3 * act_bytes),
        ("loss_pass1-3 + stats/final (ReconstructionLoss forward + backward, src/utils.py:173-241; 16 B per HR element "
         "minimum, SURVEY 8d)", k_loss, 4 * img_bytes),
    ]
    peak = float(pk["hbm_gbs"])
    out = []
    for name, fn, nbytes in cases:
        reps = 24
        for i in range(4):
            fn(i)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(reps):
                fn(i)
        graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graph.replay()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        del graph
        gbs = nbytes / (us * 1e-6) / 1e9
        out.append({"kernel": name, "bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                    "algorithmic_bytes_per_launch": nbytes, "avg_us": us})
    return out


def run_ours(a):
    import torch
    import torch.distributed as dist
    import srgan_b200 as S

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        raise SystemExit(f"--gpus {a.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    K = a.generators
    B, LH, LW = geometry(a)
    gens, opts = [], []
    for s in range(K):
        torch.manual_seed(s)
        g = S.SRResNet().to(dev)
        g.flat_parameters()
        gens.append(g)
        opts.append(S.Adam(g.parameters(), lr=1e-4, capturable=True))
    crit = S.ReconstructionLoss()
    disc, d_opt = None, None
    if a.workload == "gan-native":
        torch.manual_seed(100)
        disc = S.Discriminator().to(dev)
        disc.flat_parameters()
        d_opt = S.Adam(disc.parameters(), lr=5e-5, capturable=True)
    loss_ar = None
    if world > 1:
        S.parallel.data_parallel(gens + ([disc] if disc is not None else []), sync_batchnorm=(a.syncbn != "none"),
                                 sync_bn_transport=a.syncbn)      # "none": per-rank statistics (apportioning runs only)
        loss_ar = S.parallel.mean_over_ranks()
    policy = S.MultiGeneratorPolicy(S.PolicyConfig(num_generators=K, force=S.GAN if disc is not None else S.PIXEL, seed=0))
    use_graphs = not a.no_graphs
    trainer = S.MultiGeneratorGAN(gens, opts, crit, discriminator=disc, d_optimizer=d_opt, policy=policy,
                                  loss_allreduce=loss_ar, use_cuda_graphs=use_graphs)

    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    lr_host = torch.rand(B, 3, LH, LW, generator=gen).pin_memory()
    hr_host = torch.rand(B, 3, 4 * LH, 4 * LW, generator=gen).pin_memory()
    lr_dev, hr_dev = lr_host.to(dev), hr_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms.item())

    step_losses = [None]

    def step_resident():
        step_losses[0] = trainer.step(lr_dev, hr_dev)

    d2h_bytes = [0]
    e2e_steps = [a.steps]
    loss_host, loss_evt, last_losses = [None, None], [torch.cuda.Event(), torch.cuda.Event()], [None]
    prefetcher = [None]

    def loop_e2e():
        # the batch loop a user writes: pinned host batches -> DevicePrefetcher (copy of batch t+1 overlaps the kernels
        # of batch t; exactly one H2D copy of (hr, lr) per step, all inside the timed region) -> step -> losses to host
        # every step's losses are copied to pinned host memory right behind the step and read on the host one step
        # late (while the next step runs), like the trainer's own policy bookkeeping; the last one is read before the
        # timed region ends
        batches = ((hr_host, lr_host) for _ in range(e2e_steps[0]))
        pending = None
        if prefetcher[0] is None:
            prefetcher[0] = S.DevicePrefetcher(None, dev)      # built once, like a training script does before its epochs
        for t, (hr_d, lr_d) in enumerate(prefetcher[0].iterate(batches)):
            out = trainer.step(lr_d, hr_d)
            slot = t & 1
            if loss_host[slot] is None:
                loss_host[slot] = torch.empty(out.shape, dtype=out.dtype).pin_memory()
            loss_host[slot].copy_(out, non_blocking=True)
            loss_evt[slot].record()
            if a.e2e_sync_each_step:
                loss_evt[slot].synchronize()
                last_losses[0] = loss_host[slot].tolist()
                continue
            if pending is not None:
                loss_evt[pending].synchronize()
                last_losses[0] = loss_host[pending].tolist()          # the step's result (losses) on the host
            pending = slot
            d2h_bytes[0] = out.numel() * out.element_size()
        if pending is not None:
            loss_evt[pending].synchronize()
            last_losses[0] = loss_host[pending].tolist()

    for _ in range(max(a.warmup, 3)):
        step_resident()
    L = S.lib()
    launches0 = L.srg_total_launches()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    total_ms = timed(step_resident, a.steps)
    clocks = sampler.stop() if rank == 0 else {}
    if rank == 0 and a.dump_outputs:
        # the later legs below keep training the same models: the state is taken here, right after the timed steps
        outputs = {"losses": step_losses[0]}
        outputs.update({f"generator{i}_state": state_vector(g) for i, g in enumerate(gens)})
        if disc is not None:
            outputs["discriminator_state"] = state_vector(disc)
        dump_outputs(a.dump_outputs, outputs)
    launches = L.srg_total_launches() - launches0
    if use_graphs and trainer.launches_per_step():
        launches = trainer.launches_per_step() * a.steps      # replayed graph nodes (counted once at capture)
    ms_per_step = total_ms / a.steps
    value = world * B / (ms_per_step * 1e-3)

    # dominant kernel (3x3 64->64 conv fprop/dgrad, tcgen05): CUDA events around each launch, same stream
    trainer.use_cuda_graphs = False          # per-launch events need eagerly enqueued kernels
    for g in gens:
        g.profile_enable(True)
    prof_steps = min(a.steps, 5)
    timed(step_resident, prof_steps)
    trainer.use_cuda_graphs = use_graphs
    k_ms, k_n = 0.0, 0
    for g in gens:
        ms, n = g.profile_read()
        k_ms += ms
        k_n += n
        g.profile_enable(False)
    pk, pk_src = peaks()
    flop_per_launch = TRUNK_CONV_FLOP_PER_PIXEL * B * LH * LW
    avg_ms = k_ms / max(k_n, 1)
    achieved = flop_per_launch / (avg_ms * 1e-3) / 1e12 if k_n else 0.0
    peak = float(pk.get("bf16_tflops_sustained", pk.get("bf16_tflops")))
    peak_burst = float(pk.get("bf16_tflops", peak))
    n_layers = 1
    try:
        n_layers = max(1, int(S.lib().srg_generator_trunk_layers(gens[0].last_engine().handle)))
    except Exception:
        pass
    flop_per_launch *= n_layers            # a fused trunk launch covers 2*n_res+1 layers, a grouped launch one layer of <= 3 generators
    achieved *= n_layers
    grouped = 1 < n_layers <= 4
    traffic = None
    try:
        if not (a.workload == "cfg2" and B == 16 and LH == 96 and LW == 96):
            raise ValueError("ncu capture was taken at the cfg2 geometry")
        if n_layers != 1 and not (grouped and n_layers == 3):
            raise ValueError("captures are of the per-layer kernel and of the 3-generator grouped launch")
        fname = "r02_conv3_il_grouped_traffic.json" if grouped else "r02_conv3_il_traffic.json"
        with open(os.path.join(ROOT, "profiles", fname)) as f:
            traffic = json.load(f)["dram_bytes_per_launch"]       # dram__bytes_read.sum + dram__bytes_write.sum (ncu)
    except Exception:
        pass
    if n_layers == 1:
        kname = "conv3_il_kernel (3x3 64->64 fprop/dgrad implicit GEMM, row-interleaved N=128 tcgen05 MMAs)"
    elif grouped:
        kname = (f"conv3_il_kernel, grouped launch (the same 3x3 64->64 fprop/dgrad layer of {n_layers} generators in one launch, "
                 "row-interleaved N=128 tcgen05 MMAs)")
    else:
        kname = f"trunk_kernel (fused: {n_layers} 3x3 64->64 conv layers of one direction + their BatchNorm steps per launch)"
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "frac_of_burst_peak": achieved / peak_burst, "peak_burst": peak_burst,
                "traffic": traffic, "traffic_unit": "bytes per launch (ncu --set full, cfg2 geometry)", "kernel": kname,
                "launches_timed": k_n, "avg_launch_us": avg_ms * 1e3, "kernel_share_of_step": (k_ms / prof_steps) / ms_per_step,
                "flop_per_launch": flop_per_launch, "peak_source": pk_src + " bf16_tflops_sustained (kernel timed inside a long step)",
                "timed_over": f"{prof_steps} extra steps right after the timed region (per-launch CUDA events on the launch stream)"}
    step_flop = FLOP_PER_LR_PIXEL_FWD_BWD * B * LH * LW * K      # generator convs only (D adds ~4 % at gan-native)
    whole_step_tflops = step_flop / (ms_per_step * 1e-3) / 1e12

    e2e = None
    if not a.no_e2e:
        e2e_steps[0] = 2
        loop_e2e()
        e2e_steps[0] = a.steps
        e2e_ms = timed(loop_e2e, 1) / a.steps
        e2e = {"value": world * B / (e2e_ms * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": int(lr_host.numel() * 4 + hr_host.numel() * 4), "d2h_bytes_per_step": int(d2h_bytes[0]),
               "ms_per_step": e2e_ms, "api": "for hr, lr in DevicePrefetcher(...).iterate(pinned host batches): MultiGeneratorGAN.step(lr, hr); every step's losses copied to pinned host memory and read one step late"}
    last = trainer.step(lr_dev, hr_dev).cpu().tolist()

    # N > 1: the weak-scaling reading (16 patches per GPU, the single-GPU cfg2 batch) next to configs[2]
    weak16 = None
    if world > 1 and B != 16 and a.workload == "cfg2" and not a.no_weak16:
        lr16, hr16 = lr_dev[:16].contiguous(), hr_dev[:16].contiguous()

        def step16():
            trainer.step(lr16, hr16)
        for _ in range(3):
            step16()
        ms16 = timed(step16, a.steps) / a.steps
        weak16 = {"value": world * 16 / (ms16 * 1e-3), "unit": UNIT, "ms_per_step": ms16, "batch_per_gpu": 16,
                  "global_batch": 16 * world, "scaling": "weak"}

    hbm = None
    if rank == 0 and not a.no_hbm and a.workload == "cfg2":
        try:
            hbm = hbm_roofline(S, torch, dev, min(B, 16), LH, LW, pk)
        except Exception as exc:          # never lose the headline line to the auxiliary leg
            hbm = [{"error": str(exc)}]
    if world > 1:
        dist.barrier()

    cpu_baseline = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline and a.workload == "cfg2":
        v, dt, cores, sample, kind, bs = cpu_reference_steps(a, 2, 1)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "s_per_step": dt,
                        "sample_batch": bs}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": ("strong" if (world > 1 and a.batch is None and a.workload == "cfg2") else "weak"), "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": {"workload": workload_name(a), "generators": K, "batch_per_gpu": B, "global_batch": B * world,
                       "lr_hw": [LH, LW], "upscale": 4, "cuda_graphs": bool(use_graphs), "parallelism": f"dp{world}", "syncbn": (a.syncbn if world > 1 else None),
                       "peer_sync_timeouts": (S.parallel.peer_sync_errors() if world > 1 else 0),
                       "l2": "per-step working set (~2.5 GB of activations per generator) exceeds the 126 MB L2; no flush needed",
                       "generator_passes_per_sec": value * K,
                       "whole_step_algorithmic_tflops_per_gpu": whole_step_tflops,
                       "whole_job_algorithmic_tflops": whole_step_tflops * world,
                       "whole_step_frac_of_bf16_sustained_peak": whole_step_tflops / peak,
                       "whole_step_frac_of_bf16_burst_peak": whole_step_tflops / peak_burst,
                       "trunk_path": ("per-layer launches" if n_layers == 1 else
                                      "grouped per-layer launches (one conv launch per layer for all generators)" if grouped else
                                      "fused trunk kernel"), "last_losses": last},
            "roofline": roofline, "roofline_hbm": hbm, "weak16": weak16, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": {k: clocks.get(k) for k in ("sm_mhz", "sm_max_mhz", "reasons", "samples", "power_w_max")},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        # CUDA graphs that captured NCCL collectives are still alive: synchronise, then leave without tearing the
        # communicators down (process exit releases them; destroying them first can block)
        dist.barrier()
        torch.cuda.synchronize()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "infer-1080p":
        run_infer(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
