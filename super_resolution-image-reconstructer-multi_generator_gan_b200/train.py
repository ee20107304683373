"""Train-step functions with the reference's signatures (src/train.py:175-203, :206-230, :142-172) driving the
libsrgan_b200 modules, plus the multi-generator step the README describes (policy.py).

Differences from the reference that do not change results (SURVEY Appendix D): anomaly mode is opt-in
(``detect_anomaly``; it costs 11 % of the CPU step upstream), ``torch.cuda.empty_cache()`` is not called every step, and
the four ``.item()`` syncs are one device->host copy.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple

import torch

from .loss import tanh_mean
from .policy import GAN, PIXEL, MultiGeneratorPolicy, PolicyConfig, interpolate_models


def train_generator(generator, discriminator, lr_imgs, hr_imgs, vgg_extractor, g_criterion, g_optimizer,
                    gan_mode: bool = False, detect_anomaly: bool = False) -> Tuple[float, float, float, float]:
    """One generator update (src/train.py:175-203).  Returns (g_loss, com_loss, tv_loss, g_d_loss) as floats.

    ``gan_mode=False`` is HEAD's objective ``com_loss + tv_loss`` (src/train.py:191-192); ``gan_mode=True`` restores
    the commented-out adversarial term ``mean(tanh(D(hr) - D(sr)))`` (src/train.py:184-190).  ``vgg_extractor`` is
    accepted and ignored, as upstream."""
    losses = train_generator_async(generator, discriminator, lr_imgs, hr_imgs, vgg_extractor, g_criterion, g_optimizer,
                                   gan_mode, detect_anomaly)
    g, c, t, d = losses.tolist()           # the step's single device->host sync
    return g, c, t, d


def train_generator_async(generator, discriminator, lr_imgs, hr_imgs, vgg_extractor, g_criterion, g_optimizer,
                          gan_mode: bool = False, detect_anomaly: bool = False) -> torch.Tensor:
    """Same step, but returns the 4 losses as a device tensor [g_loss, com_loss, tv_loss, g_d_loss] without
    synchronising (lets the host run ahead; used by the multi-generator loop and bench.py)."""
    if detect_anomaly:
        torch.autograd.set_detect_anomaly(True)          # src/train.py:177
    generator.train()
    if discriminator is not None:
        discriminator.eval()                              # src/train.py:180 (no-op for InstanceNorm)
    sr_images = generator(lr_imgs)
    com_loss, tv_loss = g_criterion(hr_imgs, sr_images)
    if gan_mode:
        with discriminator.input_grad_only():             # d(D(sr))/d(sr) only; D's own .grad is never used here
            fake_preds = discriminator(sr_images)
        with torch.no_grad():
            real_preds = discriminator(hr_imgs)
        g_d_loss = tanh_mean(real_preds, fake_preds)      # mean(tanh(real - fake)), src/train.py:190
        g_loss = com_loss + tv_loss + g_d_loss
    else:
        g_d_loss = torch.zeros((), dtype=torch.float32, device=com_loss.device)   # torch.tensor(0), src/train.py:191
        g_loss = com_loss + tv_loss
    g_optimizer.zero_grad()
    g_loss.backward()
    g_optimizer.step()
    return torch.stack([g_loss.detach(), com_loss.detach(), tv_loss.detach(), g_d_loss.detach().float()])


def train_discriminator(discriminator, generator, hr_imgs, lr_imgs, d_optimizer, detect_anomaly: bool = False) -> float:
    """One discriminator update (src/train.py:206-230): ``d_loss = mean(tanh(D(G(lr)) - D(hr)))`` with G in eval mode.
    The reference keeps the autograd graph into G and throws those gradients away (SURVEY 3.2); here G's output is
    detached, which yields identical discriminator gradients."""
    return float(train_discriminator_async(discriminator, generator, hr_imgs, lr_imgs, d_optimizer, detect_anomaly))


def train_discriminator_async(discriminator, generator, hr_imgs, lr_imgs, d_optimizer,
                              detect_anomaly: bool = False) -> torch.Tensor:
    if detect_anomaly:
        torch.autograd.set_detect_anomaly(True)
    discriminator.train()
    generator.eval()
    with torch.no_grad():
        sr_imgs = generator(lr_imgs)
    # D(hr) and D(sr) as ONE pass over the concatenated batch: every op of the discriminator is per-sample
    # (InstanceNorm, no BatchNorm), so the two halves equal the reference's two separate calls (src/train.py:215-216)
    n = hr_imgs.shape[0]
    preds = discriminator(torch.cat([hr_imgs.float(), sr_imgs], dim=0))
    real_preds, fake_preds = preds[:n], preds[n:]
    d_loss = tanh_mean(fake_preds, real_preds)            # mean(tanh(fake - real)), src/train.py:218
    d_optimizer.zero_grad()
    d_loss.backward()
    d_optimizer.step()
    return d_loss.detach()


class DevicePrefetcher:
    """Host -> device staging for the batch loop (the reference copies every batch synchronously from pageable memory,
    src/train.py:152-153): wraps an iterable of (hr, lr) PINNED host tensors and yields device tensors, issuing the copy
    of batch t+1 on a side stream while the kernels of batch t run.  Two staging slots; a slot is refilled only after
    the consumer's stream has passed the point where ``release()`` was called for it."""

    def __init__(self, loader, device, depth: int = 2):
        self.loader, self.device, self.depth = loader, device, max(int(depth), 2)
        self.stream = torch.cuda.Stream(device=device)
        self.slots = [None] * self.depth
        self.ready = [torch.cuda.Event() for _ in range(self.depth)]
        self.freed = [torch.cuda.Event() for _ in range(self.depth)]

    def _stage(self, slot, batch):
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(self.freed[slot])          # no-op until the slot has been released once
            if self.slots[slot] is None:
                self.slots[slot] = [torch.empty(t.shape, dtype=t.dtype, device=self.device) for t in batch]
            for dst, src in zip(self.slots[slot], batch):
                dst.copy_(src, non_blocking=True)
            self.ready[slot].record(self.stream)

    def __iter__(self):
        return self.iterate(self.loader)

    def iterate(self, loader):
        """Iterate another loader of same-shaped batches through the SAME staging slots / stream / events (an epoch loop
        constructs the prefetcher once: no device allocation or stream creation per epoch)."""
        it = iter(loader)
        i = 0
        try:
            self._stage(0, next(it))
        except StopIteration:
            return
        while True:
            slot = i % self.depth
            try:
                self._stage((i + 1) % self.depth, next(it))   # next batch's copy overlaps this batch's kernels
                more = True
            except StopIteration:
                more = False
            torch.cuda.current_stream().wait_event(self.ready[slot])
            yield tuple(self.slots[slot])
            self.freed[slot].record(torch.cuda.current_stream())   # everything enqueued for this batch precedes the refill
            i += 1
            if not more:
                return


def train_one_epoch(generator, train_loader, g_optimizer, vgg_extractor, g_criterion, device, epoch, num_epochs,
                    discriminator, d_optimizer, prefix, verbose: bool = True) -> float:
    """Batch loop of src/train.py:142-172 (D update commented out upstream, kept off here)."""
    sums = torch.zeros(4, dtype=torch.float64)
    n = 0
    for hr_imgs, lr_imgs in train_loader:
        hr_imgs = hr_imgs.to(device, non_blocking=True)
        lr_imgs = lr_imgs.to(device, non_blocking=True)
        vals = train_generator(generator, discriminator, lr_imgs, hr_imgs, vgg_extractor, g_criterion, g_optimizer)
        sums += torch.tensor(vals, dtype=torch.float64)
        n += 1
    n = max(n, 1)
    avg = float(sums[0]) / n
    from . import parallel
    parallel.check_peer_sync()          # a SyncBatchNorm exchange that timed out during the epoch raises here
    if verbose:
        print(f"Epoch [{epoch + 1}/{num_epochs}] {prefix} Loss: {avg:.6f}")
        print(f"com_loss: {float(sums[1]) / n}, tv_loss: {float(sums[2]) / n}, g_d_loss: {float(sums[3]) / n}")
    return avg


def compute_score(generator, val_loader, device, num_batches: int = 30) -> Tuple[float, float]:
    """Validation metric of src/train.py:263-294 (called every epoch, :117): the generator in eval mode over the first
    ``num_batches`` ``(hr, lr)`` batches of ``val_loader``; returns ``(avg_psnr, avg_ssim)`` averaged over images, for this
    rank only (as upstream).  The reference scores every image on the host with calculate_psnr / calculate_ssim
    (src/utils.py:141-151); here both come from one ``image_metrics`` pass per batch, summed on the device and read back
    once.  This signature is the package's own; the generator's train / eval mode is restored and its parameters and
    BatchNorm buffers are left untouched."""
    import itertools
    from .evaluation import image_metrics
    was_training = generator.training
    generator.eval()
    sums = torch.zeros(2, dtype=torch.float64, device=device)
    images = 0
    try:
        with torch.no_grad():
            for hr_imgs, lr_imgs in itertools.islice(val_loader, num_batches):     # islice pulls no extra batch
                hr_imgs = hr_imgs.to(device, non_blocking=True)
                lr_imgs = lr_imgs.to(device, non_blocking=True)
                psnr, ssim = image_metrics(generator(lr_imgs), hr_imgs)
                sums[0] += psnr.sum()
                sums[1] += ssim.sum()
                images += hr_imgs.shape[0]
    finally:
        generator.train(was_training)
    if images == 0:
        raise ValueError("compute_score: the validation loader yielded no batch")
    avg_psnr, avg_ssim = (sums / images).tolist()          # the only device->host copy
    return avg_psnr, avg_ssim


def setup_training(rank: int, world_size: int, num_epochs: int, continue_training: bool = False, prefix: str = "Training",
                   results_dir: str = "results", num_generators: int = 1, init_process_group: bool = True,
                   capturable: bool = True):
    """The model / optimiser / scheduler set-up of the reference's ``train_example`` (src/train.py:27-71) without its
    dataset plumbing: NCCL process group on 127.0.0.1:12355 (:29-31), device = rank (:34-35), SRResNet + Discriminator
    (:45-47; data parallel through parallel.data_parallel instead of two DDP wraps), Adam with lr 1e-4 / 5e-5 (:40-41,
    61-62), ``continue_training`` resume protocol (:51-59: load rank 0's ``{prefix}_*_model_0.pth``, both LRs / 5,
    prefix "Post-Training"), LinearLR 1 -> 0.01 over ``num_epochs`` for both optimisers (:70-71).  With
    ``num_generators`` > 1 it returns the README's generator list (one optimiser / scheduler each).

    Returns a dict: generators, g_optimizers, g_schedulers, discriminator, d_optimizer, d_scheduler, g_criterion,
    device, prefix."""
    import os
    import torch.distributed as dist
    from . import parallel
    from .evaluation import load_reference_checkpoint, resume_learning_rates
    from .loss import ReconstructionLoss
    from .models import Discriminator, SRResNet
    from .optim import Adam
    if init_process_group and world_size > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "12355")
        dist.init_process_group("nccl", rank=rank, world_size=world_size)
    torch.cuda.set_device(rank)
    device = torch.device(f"cuda:{rank}")
    os.makedirs(results_dir, exist_ok=True)
    lr_generator = 1e-4
    lr_discriminator = lr_generator / 2
    g_criterion = ReconstructionLoss()
    generators = [SRResNet().to(device) for _ in range(num_generators)]
    discriminator = Discriminator().to(device)
    if continue_training:
        for i, g in enumerate(generators):
            load_reference_checkpoint(g, os.path.join(results_dir, f"{prefix}_generator_model_{0 if num_generators == 1 else i}.pth"))
        load_reference_checkpoint(discriminator, os.path.join(results_dir, f"{prefix}_discriminator_model_0.pth"))
        lr_generator, lr_discriminator = resume_learning_rates(lr_generator, lr_discriminator)
        prefix = "Post-Training"
    for m in generators + [discriminator]:
        m.flat_parameters()
    if world_size > 1:
        parallel.data_parallel(generators + [discriminator])
    g_optimizers = [Adam(g.parameters(), lr=lr_generator, capturable=capturable) for g in generators]
    d_optimizer = Adam(discriminator.parameters(), lr=lr_discriminator, capturable=capturable)
    linear = torch.optim.lr_scheduler.LinearLR
    g_schedulers = [linear(optimizer=o, start_factor=1, end_factor=0.01, total_iters=num_epochs) for o in g_optimizers]
    d_scheduler = linear(optimizer=d_optimizer, start_factor=1, end_factor=0.01, total_iters=num_epochs)
    return dict(generators=generators, g_optimizers=g_optimizers, g_schedulers=g_schedulers, discriminator=discriminator,
                d_optimizer=d_optimizer, d_scheduler=d_scheduler, g_criterion=g_criterion, device=device, prefix=prefix)


class GraphedGeneratorStep:
    """One ``train_generator`` step (forward, loss, backward, Adam) captured into a CUDA graph and replayed.

    The ~430 kernel launches of a generator step take longer to enqueue from Python than to execute on a B200; a graph
    replay is one launch.  Everything the step touches is static device memory (flat parameters / gradients / moments,
    engine workspaces, the Adam step count and learning rate as device scalars), so the replay is bit-identical to the
    eager step.  Warm-up steps needed before capture run on a side stream and are rolled back (parameters, BatchNorm
    buffers, optimiser state), so constructing this object does not train the model."""

    def __init__(self, generator, discriminator, g_criterion, g_optimizer, lr_example: torch.Tensor,
                 hr_example: torch.Tensor, gan_mode: bool = False, warmup: int = 2):
        if not getattr(g_optimizer, "capturable", False):
            raise ValueError("GraphedGeneratorStep needs optim.Adam(..., capturable=True)")
        self.generator, self.optimizer = generator, g_optimizer
        self.lr = lr_example.detach().clone()
        self.hr = hr_example.detach().clone()
        args = (generator, discriminator, self.lr, self.hr, None, g_criterion, g_optimizer, gan_mode)
        flat = generator.flat_parameters()
        rt = generator._rt
        snap = [t.clone() for t in (flat, rt["flat_buf"], rt["nbt"])]
        st0 = g_optimizer.flat_state(generator)
        opt_snap = [st0[k].clone() for k in ("m", "v", "step_dev")] if st0 is not None and "step_dev" in st0 else None
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                train_generator_async(*args)
        torch.cuda.current_stream().wait_stream(side)
        st = g_optimizer.flat_state(generator)
        with torch.no_grad():
            for dst, src in zip((flat, rt["flat_buf"], rt["nbt"]), snap):
                dst.copy_(src)
            if opt_snap is None:
                st["m"].zero_(); st["v"].zero_(); st["step_dev"].zero_()
            else:
                for k, src in zip(("m", "v", "step_dev"), opt_snap):
                    st[k].copy_(src)
        g_optimizer.zero_grad()
        torch.cuda.synchronize()
        from . import _lib
        n0 = _lib.lib().srg_total_launches()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.losses = train_generator_async(*args)
        self.launches_per_replay = int(_lib.lib().srg_total_launches() - n0)

    def __call__(self, lr_imgs: torch.Tensor, hr_imgs: torch.Tensor) -> torch.Tensor:
        """Copies the batch into the graph's static inputs, replays, returns the static [4] loss tensor (valid until
        the next call)."""
        if lr_imgs.data_ptr() != self.lr.data_ptr():
            self.lr.copy_(lr_imgs, non_blocking=True)
        if hr_imgs.data_ptr() != self.hr.data_ptr():
            self.hr.copy_(hr_imgs, non_blocking=True)
        self.optimizer.sync_lr()
        self.graph.replay()
        return self.losses


class GraphedDiscriminatorStep:
    """One ``train_discriminator`` step (generator eval forward, D forward over [hr; sr], tanh loss, D backward, Adam)
    captured into a CUDA graph; same contract as GraphedGeneratorStep (warm-up is rolled back)."""

    def __init__(self, discriminator, generator, d_optimizer, lr_example: torch.Tensor, hr_example: torch.Tensor,
                 warmup: int = 2):
        if not getattr(d_optimizer, "capturable", False):
            raise ValueError("GraphedDiscriminatorStep needs optim.Adam(..., capturable=True)")
        from . import _lib
        self.optimizer = d_optimizer
        self.lr = lr_example.detach().clone()
        self.hr = hr_example.detach().clone()
        args = (discriminator, generator, self.hr, self.lr, d_optimizer)
        flat = discriminator.flat_parameters()
        snap = flat.clone()
        st0 = d_optimizer.flat_state(discriminator)
        opt_snap = [st0[k].clone() for k in ("m", "v", "step_dev")] if st0 is not None and "step_dev" in st0 else None
        was_training = generator.training
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                train_discriminator_async(*args)
        torch.cuda.current_stream().wait_stream(side)
        st = d_optimizer.flat_state(discriminator)
        with torch.no_grad():
            flat.copy_(snap)
            if opt_snap is None:
                st["m"].zero_(); st["v"].zero_(); st["step_dev"].zero_()
            else:
                for k, src in zip(("m", "v", "step_dev"), opt_snap):
                    st[k].copy_(src)
        d_optimizer.zero_grad()
        torch.cuda.synchronize()
        n0 = _lib.lib().srg_total_launches()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.loss = train_discriminator_async(*args)
        self.launches_per_replay = int(_lib.lib().srg_total_launches() - n0)
        generator.train(was_training)

    def __call__(self, lr_imgs: torch.Tensor, hr_imgs: torch.Tensor) -> torch.Tensor:
        if lr_imgs.data_ptr() != self.lr.data_ptr():
            self.lr.copy_(lr_imgs, non_blocking=True)
        if hr_imgs.data_ptr() != self.hr.data_ptr():
            self.hr.copy_(hr_imgs, non_blocking=True)
        self.optimizer.sync_lr()
        self.graph.replay()
        return self.loss


def joint_pixel_generator_steps(generators, g_criterion, g_optimizers, lr_imgs: torch.Tensor, hr_imgs: torch.Tensor,
                                streams: Sequence[torch.cuda.Stream]) -> torch.Tensor:
    """K pixel-mode ``train_generator`` steps (src/train.py:175-203 with ``loss = com_loss + tv_loss``) on ONE batch with
    the residual trunks of all K generators executed JOINTLY: every generator runs the part of its pass before / after the
    trunk on its own stream, the trunks (16 residual blocks + conv2, forward and backward) run as one interleaved launch
    each (``srg_generators_trunk``, csrc/trunk_fused.cu), so the BatchNorm statistics latency of one generator hides
    behind the tensor work of the others.  Same arithmetic per generator as ``train_generator_async``; the autograd graph
    is bypassed (engine phases and loss kernels are called directly, ``.grad`` are views of the engines' flat gradient
    buffers).  Returns a device tensor [K, 4] of (g_loss, com_loss, tv_loss, 0) rows.  Capturable into a CUDA graph."""
    from ctypes import c_void_p
    from . import _lib
    from ._lib import check, stream_ptr
    from .loss import _scratch
    L = _lib.lib()
    K = len(generators)
    if not (1 <= K <= 4):
        raise RuntimeError("joint_pixel_generator_steps: 1..4 generators")
    lr_imgs = lr_imgs.contiguous().float()
    hr_imgs = hr_imgs.contiguous().float()
    N, _, H, W = lr_imgs.shape
    main = torch.cuda.current_stream()
    PRE, TRUNK, POST = 1, 2, 4
    engs, srs, work = [], [], []
    for i, g in enumerate(generators):
        streams[i].wait_stream(main)
        with torch.cuda.stream(streams[i]):
            g.train()
            g._flatten(lr_imgs.device)
            rt = g._rt
            eng = g._engine(N, H, W, True, lr_imgs.device, True)
            if getattr(eng, "grad_flat", None) is None:
                eng.grad_flat = torch.empty_like(rt["flat"])
            eng.bind(rt["flat"], eng.grad_flat, rt["flat_buf"])
            check(L.srg_generator_pack(eng.handle, stream_ptr()), "srg_generator_pack")
            rt["last_engine"] = eng
            if rt["nbt"] is not None and g.num_residuals > 0:
                rt["nbt"] += 1
            eng.busy = True
            sr = torch.empty(N, 3, H << g.num_upsample_stages, W << g.num_upsample_stages, dtype=torch.float32,
                             device=lr_imgs.device)
            check(L.srg_generator_forward_phases(eng.handle, c_void_p(lr_imgs.data_ptr()), c_void_p(sr.data_ptr()), 1, 1, PRE,
                                                 stream_ptr()), "srg_generator_forward_phases(pre)")
            engs.append(eng)
            srs.append(sr)
    for s_ in streams[:K]:
        main.wait_stream(s_)
    handles = (c_void_p * K)(*[e.handle for e in engs])
    check(L.srg_generators_trunk(handles, K, 0, 1, stream_ptr()), "srg_generators_trunk(forward)")
    rows = []
    for i, g in enumerate(generators):
        streams[i].wait_stream(main)
        with torch.cuda.stream(streams[i]):
            eng, sr = engs[i], srs[i]
            check(L.srg_generator_forward_phases(eng.handle, c_void_p(lr_imgs.data_ptr()), c_void_p(sr.data_ptr()), 1, 1, POST,
                                                 stream_ptr()), "srg_generator_forward_phases(post)")
            # ReconstructionLoss(hr, sr) forward + backward (src/utils.py:173-241), unit weights on both terms
            Nn, C, Hh, Ww = sr.shape
            scratch = _scratch(sr.device)
            e_buf, g_buf, dsr = torch.empty_like(sr), torch.empty_like(sr), torch.empty_like(sr)
            losses = torch.empty(2, dtype=torch.float32, device=sr.device)
            check(L.srg_recon_loss_forward(c_void_p(hr_imgs.data_ptr()), c_void_p(sr.data_ptr()), Nn, C, Hh, Ww,
                                           c_void_p(scratch.data_ptr()), scratch.numel(), c_void_p(e_buf.data_ptr()),
                                           c_void_p(g_buf.data_ptr()), c_void_p(losses.data_ptr()), stream_ptr()),
                  "srg_recon_loss_forward")
            check(L.srg_recon_loss_backward(c_void_p(hr_imgs.data_ptr()), c_void_p(sr.data_ptr()), Nn, C, Hh, Ww,
                                            c_void_p(scratch.data_ptr()), c_void_p(e_buf.data_ptr()),
                                            c_void_p(g_buf.data_ptr()), None, None, c_void_p(dsr.data_ptr()), 1.0,
                                            stream_ptr()), "srg_recon_loss_backward")
            flat_g = eng.grad_flat
            check(L.srg_generator_set_grads(eng.handle, c_void_p(flat_g.data_ptr())))
            check(L.srg_generator_backward_phases(eng.handle, c_void_p(dsr.data_ptr()), PRE, stream_ptr()),
                  "srg_generator_backward_phases(pre)")
            work.append((flat_g, losses, (scratch, e_buf, g_buf, dsr)))
    for s_ in streams[:K]:
        main.wait_stream(s_)
    check(L.srg_generators_trunk(handles, K, 1, 0, stream_ptr()), "srg_generators_trunk(backward)")
    for i, (g, o) in enumerate(zip(generators, g_optimizers)):
        streams[i].wait_stream(main)
        with torch.cuda.stream(streams[i]):
            eng = engs[i]
            flat_g, losses, _keep = work[i]
            check(L.srg_generator_backward_phases(eng.handle, None, POST, stream_ptr()), "srg_generator_backward_phases(post)")
            eng.busy = False
            g._after_backward(flat_g)                      # data-parallel gradient all-reduce hook (parallel.py)
            plist, ptable = g._rt["plist"], g._ptable
            if plist[0].grad is None or plist[0].grad.data_ptr() != flat_g.data_ptr() + 4 * ptable[0][1]:
                for p_, (_, off, n, shape) in zip(plist, ptable):      # zero_grad() dropped the views: re-attach them
                    p_.grad = flat_g[off:off + n].view(shape)
            o.step()
            zero = torch.zeros((), dtype=torch.float32, device=losses.device)
            rows.append(torch.stack([losses[0] + losses[1], losses[0], losses[1], zero]))
    for s_ in streams[:K]:
        main.wait_stream(s_)
    return torch.stack(rows)


class GraphedMultiGeneratorStep:
    """K independent pixel-mode generator steps captured as PARALLEL branches of one CUDA graph (one capture stream
    forks into K side streams and joins them again).  With ``joint=True`` (default when the fused trunk kernel applies)
    the residual trunks of the K generators run as one interleaved launch per direction (joint_pixel_generator_steps).

    The generators share nothing but the input batch, so their kernel chains may interleave: while one generator's
    persistent tensor-core kernel owns the SMs' shared memory, the HBM-bound passes (BatchNorm apply / backward,
    reductions, loss, Adam) of another generator run in the leftover thread slots instead of idling the tensor cores.
    Results are identical to running the K steps one after the other."""

    def __init__(self, generators, g_criterion, g_optimizers, lr_example: torch.Tensor, hr_example: torch.Tensor,
                 warmup: int = 2, joint: Optional[bool] = None):
        from . import _lib
        self.generators, self.optimizers = list(generators), list(g_optimizers)
        for o in self.optimizers:
            if not getattr(o, "capturable", False):
                raise ValueError("GraphedMultiGeneratorStep needs optim.Adam(..., capturable=True)")
        self.lr = lr_example.detach().clone()
        self.hr = hr_example.detach().clone()
        K = len(self.generators)
        if joint is None:
            # the joint launch pays off where the fused trunk kernel is the preferred path (see srg_set_trunk_fused);
            # warm-up falls back to per-generator branches when the engines refuse the split execution
            joint = K <= 4
        self.joint = bool(joint)
        self.streams = [torch.cuda.Stream() for _ in range(K)]
        snaps = []
        for g, o in zip(self.generators, self.optimizers):
            flat = g.flat_parameters()
            rt = g._rt
            st0 = o.flat_state(g)
            snaps.append(([t.clone() for t in (flat, rt["flat_buf"], rt["nbt"])],
                          [st0[k].clone() for k in ("m", "v", "step_dev")] if st0 is not None and "step_dev" in st0 else None))
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(max(warmup, 1)):
                if self.joint:
                    try:
                        joint_pixel_generator_steps(self.generators, g_criterion, self.optimizers, self.lr, self.hr, self.streams)
                        continue
                    except RuntimeError:
                        self.joint = False       # configuration outside the fused trunk kernel: per-generator branches
                        for g in self.generators:
                            for pool in g._rt["engines"].values():
                                for e in pool:
                                    e.busy = False
                for g, o in zip(self.generators, self.optimizers):
                    train_generator_async(g, None, self.lr, self.hr, None, g_criterion, o)
        torch.cuda.current_stream().wait_stream(side)
        with torch.no_grad():
            for g, o, (snap, osnap) in zip(self.generators, self.optimizers, snaps):
                rt = g._rt
                for dst, src in zip((rt["flat"], rt["flat_buf"], rt["nbt"]), snap):
                    dst.copy_(src)
                st = o.flat_state(g)
                if osnap is None:
                    st["m"].zero_(); st["v"].zero_(); st["step_dev"].zero_()
                else:
                    for k, src in zip(("m", "v", "step_dev"), osnap):
                        st[k].copy_(src)
                o.zero_grad()
        torch.cuda.synchronize()
        n0 = _lib.lib().srg_total_launches()
        self.graph = torch.cuda.CUDAGraph()
        rows = [None] * K
        with torch.cuda.graph(self.graph):
            if self.joint:
                self.losses = joint_pixel_generator_steps(self.generators, g_criterion, self.optimizers, self.lr, self.hr,
                                                          self.streams)
            else:
                main = torch.cuda.current_stream()
                for i, (g, o) in enumerate(zip(self.generators, self.optimizers)):
                    self.streams[i].wait_stream(main)
                    with torch.cuda.stream(self.streams[i]):
                        rows[i] = train_generator_async(g, None, self.lr, self.hr, None, g_criterion, o)
                for s_ in self.streams:
                    main.wait_stream(s_)
                self.losses = torch.stack(rows)
        self.launches_per_replay = int(_lib.lib().srg_total_launches() - n0)

    def __call__(self, lr_imgs: torch.Tensor, hr_imgs: torch.Tensor) -> torch.Tensor:
        """Replays all K steps; returns the static [K, 4] loss tensor in generator-id order."""
        if lr_imgs.data_ptr() != self.lr.data_ptr():
            self.lr.copy_(lr_imgs, non_blocking=True)
        if hr_imgs.data_ptr() != self.hr.data_ptr():
            self.hr.copy_(hr_imgs, non_blocking=True)
        for o in self.optimizers:
            o.sync_lr()
        self.graph.replay()
        return self.losses


class MultiGeneratorGAN:
    """The README's multi-generator loop (readme.md:2-10): K generators + one discriminator, loss-ranked order,
    per-generator PIXEL/GAN decision (policy.py), per-epoch re-sort.

    One ``step(lr, hr)`` = [optional discriminator update against the leader's output] + K generator updates in rank
    order.  Decisions for batch t use the running contrast losses through batch t-1, so the host never waits for
    the batch it has just enqueued (losses are read back one batch late, in one copy)."""

    def __init__(self, generators: Sequence, g_optimizers: Sequence, g_criterion, discriminator=None, d_optimizer=None,
                 policy: Optional[MultiGeneratorPolicy] = None, loss_allreduce=None, use_cuda_graphs: bool = False):
        self.generators = list(generators)
        self.g_optimizers = list(g_optimizers)
        self.criterion = g_criterion
        self.discriminator = discriminator
        self.d_optimizer = d_optimizer
        self.policy = policy or MultiGeneratorPolicy(PolicyConfig(num_generators=len(self.generators)))
        if self.policy.cfg.num_generators != len(self.generators):
            raise ValueError("policy.num_generators != len(generators)")
        self.loss_allreduce = loss_allreduce      # callable(tensor) -> None: mean over ranks, in place (parallel.py)
        self._pending: List[Tuple[List[int], torch.Tensor]] = []
        self.last_plan: List[tuple] = []
        # pixel-mode generator steps replay a captured CUDA graph per generator (built lazily on the first batch)
        self.use_cuda_graphs = use_cuda_graphs
        self._graphs: Dict[int, GraphedGeneratorStep] = {}
        self._multi: Optional[GraphedMultiGeneratorStep] = None     # all-PIXEL batches: K parallel branches, one graph
        self._d_graphs: Dict[int, "GraphedDiscriminatorStep"] = {}  # keyed by the leader generator's id
        self._gan_graphs: Dict[int, GraphedGeneratorStep] = {}

    def _drain(self, keep: int) -> None:
        while len(self._pending) > keep:
            gids, dev_losses = self._pending.pop(0)
            host = dev_losses.tolist()
            if self.loss_allreduce is not None:
                from . import parallel
                parallel.check_peer_sync()       # the host just synchronised: surface a timed-out SyncBatchNorm exchange
            for gid, row in zip(gids, host):
                self.policy.observe(gid, row[1])

    def launches_per_step(self) -> Optional[int]:
        """Kernel launches replayed per step when every generator runs from its captured graph."""
        if self._multi is not None:
            return self._multi.launches_per_replay
        graphs = list(self._graphs.values()) + list(self._gan_graphs.values()) + list(self._d_graphs.values())
        if not graphs:
            return None
        return sum(g.launches_per_replay for g in graphs)

    def step(self, lr_imgs: torch.Tensor, hr_imgs: torch.Tensor) -> torch.Tensor:
        """Returns a device tensor [K, 4] of (g_loss, com_loss, tv_loss, g_d_loss) rows in training order."""
        self._drain(keep=1)
        plan = self.policy.plan_batch()
        self.last_plan = plan
        any_gan = any(mode == GAN for _, mode in plan)
        if any_gan and self.discriminator is None:
            raise RuntimeError("the policy chose GAN mode but no discriminator was given")
        if any_gan and self.d_optimizer is not None:
            leader_id = plan[0][0]
            leader = self.generators[leader_id]
            # (data parallel: the discriminator's gradient all-reduce runs on its own library communicator and is captured
            # with the step, parallel.average_gradients_hook)
            if self.use_cuda_graphs and getattr(self.d_optimizer, "capturable", False):
                dg = self._d_graphs.get(leader_id)
                if dg is None or dg.lr.shape != lr_imgs.shape:
                    dg = GraphedDiscriminatorStep(self.discriminator, leader, self.d_optimizer, lr_imgs, hr_imgs)
                    self._d_graphs[leader_id] = dg
                dg(lr_imgs, hr_imgs)
            else:
                train_discriminator_async(self.discriminator, leader, hr_imgs, lr_imgs, self.d_optimizer)
        if self.use_cuda_graphs and not any_gan:
            if self._multi is None or self._multi.lr.shape != lr_imgs.shape:
                self._multi = GraphedMultiGeneratorStep(self.generators, self.criterion, self.g_optimizers, lr_imgs, hr_imgs)
            by_id = self._multi(lr_imgs, hr_imgs)
            gids = [gid for gid, _ in plan]
            out = by_id[gids].clone() if gids != list(range(len(gids))) else by_id.clone()
            if self.loss_allreduce is not None:
                self.loss_allreduce(out)
            self._pending.append((gids, out))
            return out
        if not any_gan and self._multi is not None and self._multi.joint and self._multi.lr.shape == lr_imgs.shape:
            # eager replay of the step the graph captured (same joint launches; used for per-launch event timing)
            by_id = joint_pixel_generator_steps(self.generators, self.criterion, self.g_optimizers, lr_imgs, hr_imgs,
                                                self._multi.streams)
            gids = [gid for gid, _ in plan]
            out = by_id[gids].clone() if gids != list(range(len(gids))) else by_id
            if self.loss_allreduce is not None:
                self.loss_allreduce(out)
            self._pending.append((gids, out))
            return out
        rows = []
        for gid, mode in plan:
            if self.use_cuda_graphs:
                cache = self._graphs if mode == PIXEL else self._gan_graphs
                gs = cache.get(gid)
                if gs is None or gs.lr.shape != lr_imgs.shape:
                    gs = GraphedGeneratorStep(self.generators[gid], self.discriminator, self.criterion,
                                              self.g_optimizers[gid], lr_imgs, hr_imgs, gan_mode=(mode == GAN))
                    cache[gid] = gs
                rows.append(gs(lr_imgs, hr_imgs).clone())
            else:
                rows.append(train_generator_async(self.generators[gid], self.discriminator, lr_imgs, hr_imgs, None,
                                                  self.criterion, self.g_optimizers[gid], gan_mode=(mode == GAN)))
        out = torch.stack(rows)
        if self.loss_allreduce is not None:
            self.loss_allreduce(out)
        self._pending.append(([gid for gid, _ in plan], out))
        return out

    def end_epoch(self) -> List[int]:
        self._drain(keep=0)
        order = self.policy.end_epoch()
        a = self.policy.cfg.lead_alpha
        if a > 0.0:
            best = self.generators[order[0]]
            for gid in order[1:]:
                interpolate_models(self.generators[gid], best, a)
        return order
