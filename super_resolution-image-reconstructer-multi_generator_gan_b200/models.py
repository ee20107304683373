"""nn.Module surface of the reference's models (reference: src/models.py) over libsrgan_b200.so.

``SRResNet`` keeps the reference's constructor signature, sub-module tree, registration order, default
initialisation (so ``torch.manual_seed(s); SRResNet()`` yields the reference's weights) and ``state_dict`` keys
(SURVEY Appendix A), but none of its arithmetic: ``forward`` / ``backward`` are single calls into the C ABI
(``srg_generator_forward`` or ``srg_generator_forward_frozen`` / ``srg_generator_backward_ex``), which enqueue
hand-written sm_100a kernels on the current CUDA stream.  There is no PyTorch / cuDNN / CPU fallback: the sub-modules below only *hold* parameters.

Parameter storage: every ``nn.Parameter`` is a view into ONE flat fp32 buffer laid out as the engine's parameter table
(``srg_generator_param_info``); gradients come back as views of one flat buffer of the same layout, so the optimiser
(``optim.Adam``) and the data-parallel gradient all-reduce are single launches over contiguous memory.
"""
from __future__ import annotations

import ctypes
import itertools
import math
import weakref
from ctypes import byref, c_char_p, c_int, c_int64, c_void_p, create_string_buffer
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib, tiling
from ._flat import _FlatModule
from ._lib import check, stream_ptr


# ----------------------------------------------------------------------------------------------------------------
# parameter holders (same registration order / default init as nn.Conv2d / nn.BatchNorm2d; never executed)
# ----------------------------------------------------------------------------------------------------------------
class _Holder(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover - guard
        raise RuntimeError(
            f"{type(self).__name__} only holds parameters; the arithmetic lives in libsrgan_b200.so and is reached "
            "through the owning SRResNet / Discriminator module (no per-layer PyTorch fallback exists)")


class ConvParams(_Holder):
    """weight [cout, cin, k, k] + bias [cout] with nn.Conv2d's default initialisation
    (kaiming_uniform(a=sqrt(5)) then U(+-1/sqrt(fan_in)) for the bias, drawn in that order)."""

    def __init__(self, cin: int, cout: int, kernel_size: int, stride: int = 1, padding: int = 0):
        super().__init__()
        self.in_channels, self.out_channels = cin, cout
        self.kernel_size, self.stride, self.padding = kernel_size, stride, padding
        self.weight = nn.Parameter(torch.empty(cout, cin, kernel_size, kernel_size))
        self.bias = nn.Parameter(torch.empty(cout))
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        bound = 1.0 / math.sqrt(cin * kernel_size * kernel_size)
        nn.init.uniform_(self.bias, -bound, bound)

    def extra_repr(self):
        return f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}, padding={self.padding}"


class BatchNormParams(_Holder):
    """nn.BatchNorm2d(C) state: weight=1, bias=0, running_mean=0, running_var=1, num_batches_tracked=0."""

    def __init__(self, channels: int, eps: float = 1e-5, momentum: float = 0.1):
        super().__init__()
        self.num_features, self.eps, self.momentum = channels, eps, momentum
        self.weight = nn.Parameter(torch.ones(channels))
        self.bias = nn.Parameter(torch.zeros(channels))
        self.register_buffer("running_mean", torch.zeros(channels))
        self.register_buffer("running_var", torch.ones(channels))
        self.register_buffer("num_batches_tracked", torch.tensor(0, dtype=torch.long))


class _Stateless(_Holder):
    """Placeholder keeping nn.Sequential indices aligned with the reference (PixelShuffle / ReLU / ... slots)."""

    def __init__(self, what: str):
        super().__init__()
        self.what = what

    def extra_repr(self):
        return self.what


class ResidualBlock(_Holder):
    """Parameter tree of the reference's ResidualBlock (src/models.py:10-25): conv1, bn1, relu, conv2, bn2.
    Executed only as part of SRResNet (the engine fuses the whole trunk)."""

    def __init__(self, num_features: int):
        super().__init__()
        self.conv1 = ConvParams(num_features, num_features, 3, padding=1)
        self.bn1 = BatchNormParams(num_features)
        self.relu = _Stateless("ReLU(inplace=True)")
        self.conv2 = ConvParams(num_features, num_features, 3, padding=1)
        self.bn2 = BatchNormParams(num_features)


# ---- engine ownership -----------------------------------------------------------------------------------------
# A grad-enabled forward marks its engine busy until backward has run.  A forward whose output is dropped WITHOUT a
# backward would otherwise keep the engine (and its multi-GB training workspace) for ever and make every such call
# allocate a new one: the autograd node's death releases it.  The token keeps a late finalizer of an OLD node (nodes
# also die after their backward) from releasing an engine that a newer forward has already re-acquired.
_busy_tokens = itertools.count(2)          # never 1: `True == 1`, and train.py marks engines with plain True


def _acquire(eng) -> int:
    eng.busy = next(_busy_tokens)
    return eng.busy


def _release_if(eng, token: int) -> None:
    if eng.busy == token:
        eng.busy = False


def _release_on_death(ctx, eng) -> None:
    ctx.busy_token = eng.busy
    weakref.finalize(ctx, _release_if, eng, eng.busy)


# ----------------------------------------------------------------------------------------------------------------
# engine wrapper
# ----------------------------------------------------------------------------------------------------------------
class _GeneratorEngine:
    """One srg_generator_t bound to a workspace: fixed (N, H, W) geometry, one in-flight forward at a time."""

    def __init__(self, N: int, H: int, W: int, n_res: int, n_up: int, training: bool, device: torch.device):
        L = _lib.lib()
        self.handle = c_void_p()
        check(L.srg_generator_create(byref(self.handle), N, H, W, n_res, n_up), "srg_generator_create")
        self.N, self.H, self.W, self.n_res, self.n_up, self.training = N, H, W, n_res, n_up, training
        self.frozen = False        # training workspace driven by srg_generator_forward_frozen (eval-mode autograd)
        self.device = device
        self.busy = False          # a training forward whose backward has not run yet
        self.ws = None
        self.bound_key = None
        self.param_elems = int(L.srg_generator_param_elems(self.handle))
        self.buffer_elems = int(L.srg_generator_buffer_elems(self.handle))

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().srg_generator_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def param_table(self) -> List[Tuple[str, int, int, Tuple[int, ...]]]:
        L = _lib.lib()
        out = []
        name = create_string_buffer(128)
        off, numel, ndim = c_int64(), c_int64(), c_int()
        shape = (c_int * 4)()
        for i in range(L.srg_generator_num_params(self.handle)):
            check(L.srg_generator_param_info(self.handle, i, name, 128, byref(off), byref(numel), byref(ndim), shape))
            out.append((name.value.decode(), off.value, numel.value, tuple(shape[k] for k in range(ndim.value))))
        return out

    def buffer_table(self) -> List[Tuple[str, int, int]]:
        L = _lib.lib()
        out = []
        name = create_string_buffer(128)
        off, numel = c_int64(), c_int64()
        for i in range(L.srg_generator_num_buffers(self.handle)):
            check(L.srg_generator_buffer_info(self.handle, i, name, 128, byref(off), byref(numel)))
            out.append((name.value.decode(), off.value, numel.value))
        return out

    def tensor_table(self) -> Dict[str, Tuple[int, Tuple[int, ...], int]]:
        L = _lib.lib()
        out = {}
        name = create_string_buffer(128)
        off, dt = c_int64(), c_int()
        dims = (c_int * 4)()
        for i in range(L.srg_generator_num_tensors(self.handle)):
            check(L.srg_generator_tensor_info(self.handle, i, name, 128, byref(off), dims, byref(dt)))
            out[name.value.decode()] = (off.value, tuple(dims[k] for k in range(4)), dt.value)
        return out

    def bind(self, flat_params: torch.Tensor, flat_grads: Optional[torch.Tensor], flat_buffers: torch.Tensor):
        L = _lib.lib()
        key = (flat_params.data_ptr(), flat_buffers.data_ptr())
        if self.ws is None:
            nbytes = int(L.srg_generator_workspace_bytes(self.handle, 1 if self.training else 0))
            self.ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
        if key != self.bound_key:
            base = self.ws.data_ptr()
            aligned = (base + 1023) & ~1023
            check(L.srg_generator_bind(self.handle, c_void_p(flat_params.data_ptr()),
                                       c_void_p(flat_grads.data_ptr()) if flat_grads is not None else None,
                                       c_void_p(flat_buffers.data_ptr()), c_void_p(aligned),
                                       self.ws.numel() - (aligned - base), 1 if self.training else 0),
                  "srg_generator_bind")
            self.ws_base = aligned
            self.bound_key = key
        elif flat_grads is not None:
            check(L.srg_generator_set_grads(self.handle, c_void_p(flat_grads.data_ptr())))

    def named_tensor(self, name: str) -> torch.Tensor:
        """bf16 NHWC intermediate inside the workspace (per-layer parity checks)."""
        off, dims, dt = self.tensor_table()[name]
        n = dims[0] * dims[1] * dims[2] * dims[3]
        start = (self.ws_base - self.ws.data_ptr()) + off
        return self.ws[start:start + 2 * n].view(torch.bfloat16).view(*dims)


class _GeneratorFn(torch.autograd.Function):
    """autograd node for one SRResNet pass: forward = srg_generator_forward (train mode) or srg_generator_forward_frozen
    (eval mode, running BatchNorm statistics), backward = srg_generator_backward_ex."""

    @staticmethod
    def forward(ctx, module, eng, lr_imgs, *params):
        L = _lib.lib()
        sr = torch.empty(eng.N, 3, eng.H << eng.n_up, eng.W << eng.n_up, dtype=torch.float32, device=lr_imgs.device)
        if eng.frozen:
            check(L.srg_generator_forward_frozen(eng.handle, c_void_p(lr_imgs.data_ptr()), c_void_p(sr.data_ptr()),
                                                 stream_ptr()), "srg_generator_forward_frozen")
        else:
            check(L.srg_generator_forward(eng.handle, c_void_p(lr_imgs.data_ptr()), c_void_p(sr.data_ptr()),
                                          1 if module.training else 0, 1 if module.training else 0, stream_ptr()),
                  "srg_generator_forward")
        ctx.module_ref = weakref.ref(module)
        ctx.x_shape = tuple(lr_imgs.shape)
        ctx.eng = eng
        _release_on_death(ctx, eng)
        ctx.n_params = len(params)
        ctx.set_materialize_grads(False)
        return sr

    @staticmethod
    def backward(ctx, dsr):
        module = ctx.module_ref()
        eng = ctx.eng
        if dsr is None or module is None:
            _release_if(eng, ctx.busy_token)
            return (None,) * (3 + ctx.n_params)
        L = _lib.lib()
        dsr = dsr.contiguous()
        if dsr.dtype != torch.float32:
            dsr = dsr.float()
        # data-parallel ranks take the same branch: their requires_grad flags are identical
        want_dx = ctx.needs_input_grad[2]
        want_pg = any(ctx.needs_input_grad[3:])
        dlr = torch.empty(ctx.x_shape, dtype=torch.float32, device=dsr.device) if want_dx else None
        flat_g = None
        if want_pg:
            flat_g = module._grad_buffer_for_backward(eng)
            check(L.srg_generator_set_grads(eng.handle, c_void_p(flat_g.data_ptr())))
        check(L.srg_generator_backward_ex(eng.handle, c_void_p(dsr.data_ptr()), 1 if want_pg else 0,
                                          c_void_p(dlr.data_ptr()) if dlr is not None else None, stream_ptr()),
              "srg_generator_backward_ex")
        _release_if(eng, ctx.busy_token)
        if not want_pg:
            # input gradient only: the flat gradient buffer, the gradient hook and .grad are left alone
            return (None, None, dlr) + (None,) * ctx.n_params
        module._after_backward(flat_g)
        grads = tuple(flat_g[off:off + n].view(shape) for (_, off, n, shape) in module._ptable)
        return (None, None, dlr) + grads


class _FrozenTilesFn(torch.autograd.Function):
    """autograd node of an eval-mode forward under ``SRResNet.grad_budget_bytes``: the frozen forward of every window
    (``srg_generator_forward_frozen_tiles``), call by call through one engine of ``n`` windows.  The engine keeps only the
    last call's activations, so the backward recomputes each call's windows before running their backward
    (``srg_generator_backward_tiles``).  Each backward recomputes its own windows, so the engine is not reserved between
    forward and backward and any number of such graphs can be alive at once."""

    @staticmethod
    def forward(ctx, module, plan, x, *params):
        win_h, win_w, n, tiles = plan
        s = module.num_upsample_stages
        eng = module._frozen_tiles_engine(n, win_h, win_w, x.device)
        sr = torch.empty(x.shape[0], 3, x.shape[2] << s, x.shape[3] << s, dtype=torch.float32, device=x.device)
        for i in range(0, len(tiles), n):
            tiling.forward_frozen_tiles(eng.handle, x, tiles[i:i + n], sr, stream_ptr())
        ctx.save_for_backward(x)
        ctx.module_ref = weakref.ref(module)
        ctx.plan = plan
        ctx.versions = module._state_versions()
        ctx.n_params = len(params)
        ctx.set_materialize_grads(False)
        return sr

    @staticmethod
    def backward(ctx, dsr):
        module = ctx.module_ref()
        if dsr is None or module is None:
            return (None,) * (3 + ctx.n_params)
        (x,) = ctx.saved_tensors
        if module._state_versions() != ctx.versions:
            raise RuntimeError("SRResNet: a parameter or BatchNorm buffer was modified in place between the forward and the "
                               "backward of an eval-mode forward under grad_budget_bytes (its backward recomputes the "
                               "forward from the current values)")
        dsr = dsr.contiguous()
        if dsr.dtype != torch.float32:
            dsr = dsr.float()
        want_dx = ctx.needs_input_grad[2]
        want_pg = any(ctx.needs_input_grad[3:])
        win_h, win_w, n, tiles = ctx.plan
        eng = module._frozen_tiles_engine(n, win_h, win_w, x.device)       # re-packs the weights
        dlr = torch.zeros(x.shape, dtype=torch.float32, device=x.device) if want_dx else None
        total = module._grad_buffer_for_backward(eng) if want_pg else None
        part = torch.empty_like(total) if want_pg and len(tiles) > n else None
        L = _lib.lib()
        for k, i in enumerate(range(0, len(tiles), n)):
            tiling.forward_frozen_tiles(eng.handle, x, tiles[i:i + n], None, stream_ptr())
            if want_pg:
                # the first call writes the running total, later ones a second buffer that is added to it
                check(L.srg_generator_set_grads(eng.handle, c_void_p((total if k == 0 else part).data_ptr())))
            tiling.backward_tiles(eng.handle, dsr, want_pg, dlr, stream_ptr())
            if want_pg and k > 0:
                total.add_(part)
        if not want_pg:
            # input gradient only: the flat gradient buffer, the gradient hook and .grad are left alone
            return (None, None, dlr) + (None,) * ctx.n_params
        module._after_backward(total)
        grads = tuple(total[off:off + m].view(shape) for (_, off, m, shape) in module._ptable)
        return (None, None, dlr) + grads


class SRResNet(_FlatModule):
    """Drop-in for the reference's SRResNet (src/models.py:44-87).

    conv 9x9 (3->64) + LeakyReLU(0.2) -> ``num_residuals`` x [conv3x3, BN, ReLU, conv3x3, BN, +skip] -> conv3x3 ->
    + global skip -> ``int(upscale_factor // 2)`` x [conv3x3 (64->256), PixelShuffle(2), ReLU] -> conv 9x9 (64->3).
    Input / output: NCHW fp32 CUDA tensors; ``upscale_u8`` takes and returns uint8 NHWC frames.  The kernels are specialised for in_channels=3, num_features=64 (the
    reference's only configuration); other widths raise.
    """

    def __init__(self, in_channels: int = 3, num_features: int = 64, num_residuals: int = 16, upscale_factor: int = 4):
        super().__init__()
        if in_channels != 3 or num_features != 64:
            raise NotImplementedError("libsrgan_b200 implements the reference configuration in_channels=3, num_features=64")
        self.in_channels, self.num_features = in_channels, num_features
        self.num_residuals = num_residuals
        self.num_upsample_stages = int(upscale_factor // 2)      # reference quirk: 2->1, 3->1, 4->2, 8->4 stages
        self.conv1 = ConvParams(in_channels, num_features, 9, padding=4)
        self.relu = _Stateless("LeakyReLU(0.2, inplace=True)")
        self.residual_blocks = nn.Sequential(*[ResidualBlock(num_features) for _ in range(num_residuals)])
        self.conv2 = ConvParams(num_features, num_features, 3, padding=1)
        ups: List[nn.Module] = []
        for _ in range(self.num_upsample_stages):
            ups += [ConvParams(num_features, num_features * 4, 3, padding=1), _Stateless("PixelShuffle(2)"),
                    _Stateless("ReLU(inplace=True)")]
        self.upsample = nn.Sequential(*ups)
        self.conv3 = ConvParams(num_features, in_channels, 9, padding=4)
        self._reset_runtime()

    def _probe_engine(self, device) -> _GeneratorEngine:
        rt = self._rt
        if rt.get("probe") is None:
            rt["probe"] = _GeneratorEngine(1, 8, 8, self.num_residuals, self.num_upsample_stages, False, device)
        return rt["probe"]

    def _tables(self, device):
        probe = self._probe_engine(device)
        return probe.param_table(), probe.buffer_table(), probe.param_elems, probe.buffer_elems

    # ---- engines ---------------------------------------------------------------------------------------------------
    def _engine(self, N: int, H: int, W: int, training: bool, device, need_grad: bool,
                frozen: bool = False) -> _GeneratorEngine:
        rt = self._rt
        # frozen engines (eval-mode autograd) run on a training-sized workspace but in their own pool
        key = (N, H, W, "frozen") if frozen else (N, H, W, training)
        pool = rt["engines"].setdefault(key, [])
        eng = None
        for e in pool:
            if not e.busy:
                eng = e
                break
        if eng is None:
            eng = _GeneratorEngine(N, H, W, self.num_residuals, self.num_upsample_stages, training or frozen, device)
            eng.frozen = frozen
            if rt["sync_bn"]:
                self._attach_sync_bn(eng)
            if getattr(self, "debug_keep_grads", False):
                check(_lib.lib().srg_generator_set_keep_grads(eng.handle, 1))
            if rt.get("profile"):
                check(_lib.lib().srg_generator_profile_enable(eng.handle, 1))
            pool.append(eng)
        return eng

    def _attach_sync_bn(self, eng):
        kind, obj, world = self._rt["sync_bn"]
        if kind == "peer":
            check(_lib.lib().srg_generator_use_peer_sync(eng.handle, obj), "srg_generator_use_peer_sync")
        else:
            check(_lib.lib().srg_generator_use_nccl(eng.handle, obj, world), "srg_generator_use_nccl")

    def enable_sync_batchnorm(self, comm=None, world: int = 1, peer_sync=None):
        """SyncBatchNorm: per-channel sums are reduced across ranks between the local reduction and the BatchNorm
        finalize, forward and backward -- through ``peer_sync`` (parallel.create_peer_sync(): NVLink peer-memory
        exchange fused with the finalize kernel) or an NCCL communicator (parallel.create_comm())."""
        self._rt["sync_bn"] = ("peer", peer_sync, int(world)) if peer_sync is not None else ("nccl", comm, int(world))
        for pool in self._rt["engines"].values():
            for e in pool:
                self._attach_sync_bn(e)

    def launch_count(self) -> int:
        L = _lib.lib()
        return sum(int(L.srg_generator_launch_count(e.handle)) for pool in self._rt["engines"].values() for e in pool)

    def profile_enable(self, on: bool = True) -> None:
        """CUDA-event timing of the dominant kernel class (3x3 64->64 conv fprop/dgrad launches), see bench.py."""
        self._rt["profile"] = bool(on)
        for pool in self._rt["engines"].values():
            for e in pool:
                check(_lib.lib().srg_generator_profile_enable(e.handle, 1 if on else 0))

    def profile_read(self) -> Tuple[float, int]:
        """(summed device ms, launches) of the profiled kernel class since the last read."""
        from ctypes import c_double, c_longlong
        total, count = 0.0, 0
        for pool in self._rt["engines"].values():
            for e in pool:
                ms, n = c_double(), c_longlong()
                check(_lib.lib().srg_generator_profile_read(e.handle, byref(ms), byref(n)), "profile_read")
                total += ms.value
                count += n.value
        return total, count

    def last_engine(self) -> Optional[_GeneratorEngine]:
        return self._rt["last_engine"]

    #: eval-mode activation budget in bytes: larger batches are streamed in chunks of frames (None: never chunk)
    stream_budget_bytes: Optional[int] = 6 << 30

    #: eval-mode workspace budget in bytes for ONE frame: a frame whose whole-frame eval workspace is larger is upscaled
    #: window by window (spatial tiles with a halo, ``tiling.plan_tiles``), bit-identical to the whole-frame forward,
    #: with at most this much engine workspace (None: never tile)
    tile_budget_bytes: Optional[int] = None

    def _eval_ws_bytes(self, H: int, W: int, device) -> int:
        """eval workspace of a one-frame H x W engine (a probe engine: creation needs no device memory)"""
        rt = self._rt
        key = ("ws1", H, W)
        if key not in rt:
            probe = _GeneratorEngine(1, H, W, self.num_residuals, self.num_upsample_stages, False, device)
            rt[key] = int(_lib.lib().srg_generator_workspace_bytes(probe.handle, 0))
            del probe
        return rt[key]

    def _stream_chunk(self, N: int, H: int, W: int, device) -> int:
        """Frames per eval-mode engine call such that the engine workspace stays within ``stream_budget_bytes``."""
        budget = self.stream_budget_bytes
        if budget is None:
            return N
        per_frame = max(self._eval_ws_bytes(H, W, device), 1)
        return max(1, min(N, int(budget // per_frame)))

    #: eval-mode autograd workspace budget in bytes: an eval forward whose input requires grad, and whose whole-batch
    #: frozen (training-layout) workspace is larger, runs in halo-padded windows (``tiling.plan_tiles``; a frame that fits
    #: is one window) through one engine of at most this much workspace, and its backward recomputes the windows' forward
    #: (None: the whole batch in one engine call)
    grad_budget_bytes: Optional[int] = None

    def _train_ws_bytes(self, N: int, H: int, W: int, device) -> int:
        """training (frozen) workspace of an N x H x W engine, as ``_engine`` would create it (a host-only probe)"""
        rt = self._rt
        keep = bool(getattr(self, "debug_keep_grads", False))
        key = ("ws_train", N, H, W, keep)
        if key not in rt:
            probe = _GeneratorEngine(N, H, W, self.num_residuals, self.num_upsample_stages, True, device)
            if keep:
                check(_lib.lib().srg_generator_set_keep_grads(probe.handle, 1))
            rt[key] = int(_lib.lib().srg_generator_workspace_bytes(probe.handle, 1))
            del probe
        return rt[key]

    def _state_versions(self) -> Tuple[int, ...]:
        return tuple(p._version for p in self._rt["plist"]) + tuple(b._version for b in self.buffers())

    def _frozen_tiles_engine(self, n: int, H: int, W: int, device) -> _GeneratorEngine:
        """a frozen engine of n windows of H x W, bound and with freshly packed weights"""
        rt = self._rt
        eng = self._engine(n, H, W, False, device, False, frozen=True)
        if getattr(eng, "grad_flat", None) is None:
            eng.grad_flat = torch.empty_like(rt["flat"])
        eng.bind(rt["flat"], eng.grad_flat, rt["flat_buf"])
        check(_lib.lib().srg_generator_pack(eng.handle, stream_ptr()), "srg_generator_pack")
        rt["last_engine"] = eng
        return eng

    def _frozen_tiles_plan(self, N: int, H: int, W: int, device) -> Tuple[int, int, int, list]:
        """(window_h, window_w, windows per call, windows) for ``grad_budget_bytes``: the planner's windows, and as many
        per call as an engine of that many windows fits the budget"""
        rt = self._rt
        budget = int(self.grad_budget_bytes)
        key = ("frozen_tiles", N, H, W, budget, bool(getattr(self, "debug_keep_grads", False)))
        if key not in rt:
            halo = tiling.tile_halo(self.num_residuals, self.num_upsample_stages)
            win_h, win_w, per_call, tiles = tiling.plan_tiles(N, H, W, halo,
                                                              lambda h, w: self._train_ws_bytes(1, h, w, device), budget)
            n = min(per_call, len(tiles))
            while n > 1 and self._train_ws_bytes(n, win_h, win_w, device) > budget:
                n -= 1
            rt[key] = (win_h, win_w, n, tiles)
        return rt[key]

    def _forward_tiled(self, x: torch.Tensor, u8: bool = False) -> torch.Tensor:
        """eval-mode forward of frames too large for ``tile_budget_bytes``: the windows of all frames in order, as many per
        ``srg_generator_forward_tiles`` call as the plan's ``tiles_per_call`` (usually 1: the planner picks the largest
        window that fits), through ONE engine of that many windows.  ``u8``: uint8 N x H x W x 3 frames in and out
        (``upscale_u8``, ``srg_generator_forward_tiles_u8``), with the same plan and engine."""
        N, H, W = (x.shape[0], x.shape[1], x.shape[2]) if u8 else (x.shape[0], x.shape[2], x.shape[3])
        rt = self._rt
        budget = int(self.tile_budget_bytes)
        key = ("tiles", N, H, W, budget)
        if key not in rt:
            halo = tiling.tile_halo(self.num_residuals, self.num_upsample_stages)
            rt[key] = tiling.plan_tiles(N, H, W, halo, lambda h, w: self._eval_ws_bytes(h, w, x.device), budget)
        win_h, win_w, per_call, tiles = rt[key]
        s = self.num_upsample_stages
        if u8:
            sr = torch.empty(N, H << s, W << s, 3, dtype=torch.uint8, device=x.device)
        else:
            sr = torch.empty(N, 3, H << s, W << s, dtype=torch.float32, device=x.device)
        n = min(per_call, len(tiles))
        eng = self._engine(n, win_h, win_w, False, x.device, False)
        eng.bind(rt["flat"], None, rt["flat_buf"])
        check(_lib.lib().srg_generator_pack(eng.handle, stream_ptr()), "srg_generator_pack")
        rt["last_engine"] = eng
        call = tiling.forward_tiles_u8 if u8 else tiling.forward_tiles
        for i in range(0, len(tiles), n):
            call(eng.handle, x, tiles[i:i + n], sr, stream_ptr())
        return sr

    # ---- forward ---------------------------------------------------------------------------------------------------
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """N x 3 x H x W fp32 CUDA -> N x 3 x (H << s) x (W << s), s = ``num_upsample_stages``.

        ====== ========= ================== ========================= =================================================
        mode   grad mode ``x.requires_grad`` any param requires grad   behaviour
        ====== ========= ================== ========================= =================================================
        train  on        no                 any                       batch statistics; parameter gradients
        train  on        yes                yes                       the same, plus ``x.grad``
        train  on        yes                no                        input-only backward: ``x.grad``, no parameter
                                                                      gradient is computed and the gradient hook is
                                                                      not called
        eval   off       any                any                       detached output, BatchNorm folded into the convs,
                                                                      large batches streamed in chunks
        eval   off       any                any                       with ``tile_budget_bytes`` set and a frame whose
                                                                      eval workspace exceeds it: every frame upscaled
                                                                      in spatial windows with a halo (the largest
                                                                      window that fits, so usually one window per
                                                                      engine call), bit-identical
        eval   on        no                 any                       the same (detached)
        eval   on        yes                any                       running BatchNorm statistics, never updated
                                                                      ("frozen"), whole batch in one engine call:
                                                                      ``x.grad`` plus the gradients of the parameters
                                                                      that require grad
        eval   on        yes                any                       with ``grad_budget_bytes`` set and a whole-batch
                                                                      frozen workspace above it: the same gradients,
                                                                      summed over halo-padded windows (a frame that
                                                                      fits is one window) run through one engine within
                                                                      the budget; the backward recomputes each call's
                                                                      windows; equal to the whole-batch path up to
                                                                      fp32 summation order and bf16 rounding
        ====== ========= ================== ========================= =================================================

        The frozen output equals the detached eval output up to bf16 rounding (DESIGN §4).  Double backward is not
        supported.
        """
        if not x.is_cuda:
            raise RuntimeError("SRResNet (libsrgan_b200) runs on a CUDA device only; there is no CPU path")
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError(f"expected an N x 3 x H x W input, got {tuple(x.shape)}")
        x = x.contiguous()
        if x.dtype != torch.float32:
            x = x.float()
        N, _, H, W = x.shape
        self._flatten(x.device)
        rt = self._rt
        need_grad = self.training and torch.is_grad_enabled()
        # eval mode with an input that requires grad (a fixed generator inside a larger differentiable pipeline)
        frozen = not self.training and torch.is_grad_enabled() and x.requires_grad
        if (frozen and self.grad_budget_bytes is not None
                and self._train_ws_bytes(N, H, W, x.device) > self.grad_budget_bytes):
            return _FrozenTilesFn.apply(self, self._frozen_tiles_plan(N, H, W, x.device), x, *rt["plist"])
        if (not self.training and not frozen and self.tile_budget_bytes is not None
                and self._eval_ws_bytes(H, W, x.device) > self.tile_budget_bytes):
            return self._forward_tiled(x)
        if not self.training and N > 1 and not frozen:
            # Evaluation (src/evaluation.py:48-50, BASELINE configs[3]): frames are independent in eval mode (running
            # BatchNorm statistics), so a batch whose activations would not fit the streaming budget is run in chunks
            # of whole frames through ONE smaller engine: peak memory is O(chunk), the arithmetic per frame (and hence
            # every output bit) is that of the unchunked call.  8 x 1080p would otherwise materialise ~34 GB.
            chunk = self._stream_chunk(N, H, W, x.device)
            if chunk < N:
                sr = torch.empty(N, 3, H << self.num_upsample_stages, W << self.num_upsample_stages, dtype=torch.float32,
                                 device=x.device)
                packed = set()                             # engines whose bf16 weight copy is current for THIS call
                for i in range(0, N, chunk):
                    j = min(N, i + chunk)
                    self._eval_into(x[i:j], sr[i:j], packed)   # whole frames of an NCHW batch are contiguous: no copy
                return sr
        eng = self._engine(N, H, W, self.training, x.device, need_grad, frozen=frozen)
        if eng.training and getattr(eng, "grad_flat", None) is None:
            eng.grad_flat = torch.empty_like(rt["flat"])
        eng.bind(rt["flat"], eng.grad_flat if eng.training else None, rt["flat_buf"])
        L = _lib.lib()
        check(L.srg_generator_pack(eng.handle, stream_ptr()), "srg_generator_pack")
        rt["last_engine"] = eng
        if self.training and rt["nbt"] is not None and self.num_residuals > 0:
            rt["nbt"] += 1
        if need_grad or frozen:
            _acquire(eng)
            return _GeneratorFn.apply(self, eng, x, *rt["plist"])
        # eval mode (running statistics) or no_grad: no autograd graph.  The reference keeps a graph through an
        # eval-mode generator in train_discriminator (src/train.py:212) but discards those gradients (SURVEY 3.2).
        sr = torch.empty(N, 3, H << self.num_upsample_stages, W << self.num_upsample_stages, dtype=torch.float32,
                         device=x.device)
        check(L.srg_generator_forward(eng.handle, c_void_p(x.data_ptr()), c_void_p(sr.data_ptr()),
                                      1 if self.training else 0, 1 if self.training else 0, stream_ptr()),
              "srg_generator_forward")
        return sr

    def _eval_into(self, x: torch.Tensor, out: torch.Tensor, packed: set) -> None:
        """eval-mode forward of a chunk of frames straight into ``out`` (a contiguous slice of the caller's batch): fp32
        NCHW, or uint8 NHWC in and out (``upscale_u8``, ``srg_generator_forward_u8``)."""
        assert x.is_contiguous() and out.is_contiguous()
        u8 = x.dtype == torch.uint8
        n, H, W = (x.shape[0], x.shape[1], x.shape[2]) if u8 else (x.shape[0], x.shape[2], x.shape[3])
        rt = self._rt
        eng = self._engine(n, H, W, False, x.device, False)
        eng.bind(rt["flat"], None, rt["flat_buf"])
        L = _lib.lib()
        if id(eng) not in packed:
            check(L.srg_generator_pack(eng.handle, stream_ptr()), "srg_generator_pack")
            packed.add(id(eng))
        rt["last_engine"] = eng
        if u8:
            check(L.srg_generator_forward_u8(eng.handle, c_void_p(x.data_ptr()), c_void_p(out.data_ptr()), stream_ptr()),
                  "srg_generator_forward_u8")
            return
        check(L.srg_generator_forward(eng.handle, c_void_p(x.data_ptr()), c_void_p(out.data_ptr()), 0, 0, stream_ptr()),
              "srg_generator_forward")

    def upscale_u8(self, frames: torch.Tensor) -> torch.Tensor:
        """8-bit frames in and out: uint8 N x H x W x 3 CUDA (decoded RGB, channel-last, as ``transformers`` takes
        them) -> uint8 N x (H << s) x (W << s) x 3, s = ``num_upsample_stages``.

        The result is, bit for bit, ``q(self(transformers.to_tensor(frames)))`` with
        ``q(sr) = (sr.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1)``: conv1 reads each byte v as
        v / 255 with ToTensor's fp32 division, and conv3's epilogue stores round-half-even(255 * clamp(y, 0, 1)).  Neither
        an fp32 copy of the input nor an fp32 SR tensor is made.  A NaN output stores 0 (torch's cast of NaN is
        undefined).  Eval mode only.  Frames are routed like the detached eval forward: streamed in chunks under
        ``stream_budget_bytes``, upscaled in windows under ``tile_budget_bytes``, through the same engines.  No autograd
        graph is built.
        """
        if self.training:
            raise RuntimeError("SRResNet.upscale_u8 runs the eval forward only: call .eval() first")
        if frames.dtype != torch.uint8:
            raise RuntimeError(f"SRResNet.upscale_u8 takes uint8 frames, got {frames.dtype}")
        if frames.dim() != 4 or frames.shape[3] != 3 or min(frames.shape) < 1:
            raise RuntimeError(f"SRResNet.upscale_u8 expects an N x H x W x 3 batch, got {tuple(frames.shape)}")
        if not frames.is_cuda:
            raise RuntimeError("SRResNet.upscale_u8 (libsrgan_b200) takes a CUDA tensor; there is no CPU path")
        frames = frames.contiguous()
        N, H, W, _ = frames.shape
        self._flatten(frames.device)
        if self.tile_budget_bytes is not None and self._eval_ws_bytes(H, W, frames.device) > self.tile_budget_bytes:
            return self._forward_tiled(frames, u8=True)
        s = self.num_upsample_stages
        sr = torch.empty(N, H << s, W << s, 3, dtype=torch.uint8, device=frames.device)
        chunk = self._stream_chunk(N, H, W, frames.device) if N > 1 else N
        packed = set()
        for i in range(0, N, chunk):
            j = min(N, i + chunk)
            self._eval_into(frames[i:j], sr[i:j], packed)
        return sr


# ----------------------------------------------------------------------------------------------------------------
# Discriminator
# ----------------------------------------------------------------------------------------------------------------
class _DiscriminatorEngine:
    """One srg_discriminator_t bound to a workspace: fixed (N, H, W) geometry, one in-flight forward at a time."""

    def __init__(self, N: int, H: int, W: int, training: bool, device):
        L = _lib.lib()
        self.handle = c_void_p()
        rc = L.srg_discriminator_create(byref(self.handle), N, H, W)
        if rc != 0:
            msg = L.srg_last_error()
            # same failure mode as the reference (a RuntimeError out of MaxPool2d / InstanceNorm2d, SURVEY Appendix E)
            raise RuntimeError(msg.decode() if msg else f"srg_discriminator_create failed ({rc})")
        self.N, self.H, self.W, self.training, self.device = N, H, W, training, device
        self.busy = False
        self.ws = None
        self.bound_key = None
        self.param_elems = int(L.srg_discriminator_param_elems(self.handle))
        oh, ow = c_int(), c_int()
        L.srg_discriminator_output_hw(self.handle, byref(oh), byref(ow))
        self.out_hw = (oh.value, ow.value)

    def __del__(self):
        try:
            if self.handle:
                _lib.lib().srg_discriminator_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    def param_table(self):
        L = _lib.lib()
        out = []
        name = create_string_buffer(128)
        off, numel, ndim = c_int64(), c_int64(), c_int()
        shape = (c_int * 4)()
        for i in range(L.srg_discriminator_num_params(self.handle)):
            check(L.srg_discriminator_param_info(self.handle, i, name, 128, byref(off), byref(numel), byref(ndim), shape))
            out.append((name.value.decode(), off.value, numel.value, tuple(shape[k] for k in range(ndim.value))))
        return out

    def tensor_table(self):
        L = _lib.lib()
        out = {}
        name = create_string_buffer(128)
        off, dt = c_int64(), c_int()
        dims = (c_int * 4)()
        for i in range(L.srg_discriminator_num_tensors(self.handle)):
            check(L.srg_discriminator_tensor_info(self.handle, i, name, 128, byref(off), dims, byref(dt)))
            out[name.value.decode()] = (off.value, tuple(dims[k] for k in range(4)), dt.value)
        return out

    def bind(self, flat_params: torch.Tensor, flat_grads: Optional[torch.Tensor]):
        L = _lib.lib()
        key = flat_params.data_ptr()
        if self.ws is None:
            nbytes = int(L.srg_discriminator_workspace_bytes(self.handle, 1 if self.training else 0))
            self.ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=self.device)
        if key != self.bound_key:
            base = self.ws.data_ptr()
            aligned = (base + 1023) & ~1023
            check(L.srg_discriminator_bind(self.handle, c_void_p(flat_params.data_ptr()),
                                           c_void_p(flat_grads.data_ptr()) if flat_grads is not None else None,
                                           c_void_p(aligned), self.ws.numel() - (aligned - base), 1 if self.training else 0),
                  "srg_discriminator_bind")
            self.ws_base = aligned
            self.bound_key = key

    def named_tensor(self, name: str) -> torch.Tensor:
        off, dims, dt = self.tensor_table()[name]
        n = dims[0] * dims[1] * dims[2] * dims[3]
        start = (self.ws_base - self.ws.data_ptr()) + off
        if dt == 0:
            return self.ws[start:start + 2 * n].view(torch.bfloat16).view(*dims)
        return self.ws[start:start + 4 * n].view(torch.float32).view(*dims)


class _DiscriminatorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, eng, x, *params):
        L = _lib.lib()
        out = torch.empty(eng.N, 512, eng.out_hw[0], eng.out_hw[1], dtype=torch.float32, device=x.device)
        check(L.srg_discriminator_forward(eng.handle, c_void_p(x.data_ptr()), c_void_p(out.data_ptr()), stream_ptr()),
              "srg_discriminator_forward")
        ctx.module_ref = weakref.ref(module)
        ctx.eng = eng
        _release_on_death(ctx, eng)
        ctx.n_params = len(params)
        ctx.x_shape = tuple(x.shape)
        ctx.param_grads = module._rt.get("param_grads", True)
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, dout):
        module = ctx.module_ref()
        eng = ctx.eng
        if dout is None or module is None:
            _release_if(eng, ctx.busy_token)
            return (None,) * (3 + ctx.n_params)
        L = _lib.lib()
        dout = dout.contiguous()
        if dout.dtype != torch.float32:
            dout = dout.float()
        want_dx = ctx.needs_input_grad[2]
        want_pg = ctx.param_grads and any(ctx.needs_input_grad[3:])
        dx = torch.empty(ctx.x_shape, dtype=torch.float32, device=dout.device) if want_dx else None
        flat_g = None
        if want_pg:
            flat_g = module._grad_buffer_for_backward(eng)
            check(L.srg_discriminator_set_grads(eng.handle, c_void_p(flat_g.data_ptr())))
        check(L.srg_discriminator_backward(eng.handle, c_void_p(dout.data_ptr()), 1 if want_pg else 0,
                                           c_void_p(dx.data_ptr()) if dx is not None else None, stream_ptr()),
              "srg_discriminator_backward")
        _release_if(eng, ctx.busy_token)
        if want_pg:
            module._after_backward(flat_g)
            grads = tuple(flat_g[off:off + n].view(shape) for (_, off, n, shape) in module._ptable)
        else:
            grads = (None,) * ctx.n_params
        return (None, None, dx) + grads


class Discriminator(_FlatModule):
    """Drop-in for the reference's Discriminator (src/models.py:90-120): ``self.model`` is an nn.Sequential whose
    indices 0, 4, 8, 12 hold the conv parameters (state_dict keys ``model.0.weight`` ...).  Input N x 3 x H x W fp32
    CUDA -> N x 512 x h x w sigmoid map.  Raises RuntimeError for inputs the reference network cannot process (every
    axis must be >= 428 and one >= 684, SURVEY Appendix E)."""

    def __init__(self, input_channels: int = 3, num_filters: int = 64):
        super().__init__()
        if input_channels != 3 or num_filters != 64:
            raise NotImplementedError("libsrgan_b200 implements the reference configuration input_channels=3, num_filters=64")
        nf = num_filters
        layers: List[nn.Module] = []
        specs = [(input_channels, nf, 8, 2), (nf, nf * 2, 4, 1), (nf * 2, nf * 4, 4, 1), (nf * 4, nf * 8, 4, 1)]
        for i, (cin, cout, k, pad) in enumerate(specs):
            layers += [ConvParams(cin, cout, k, stride=2, padding=pad), _Stateless("MaxPool2d(kernel_size=3, stride=2)"),
                       _Stateless(f"InstanceNorm2d({cout})")]
            layers.append(_Stateless("LeakyReLU(0.2)") if i < 3 else _Stateless("Sigmoid()"))
        self.model = nn.Sequential(*layers)
        self._reset_runtime()

    def _tables(self, device):
        rt = self._rt
        if rt.get("probe") is None:
            rt["probe"] = _DiscriminatorEngine(1, 428, 684, False, device)
        probe = rt["probe"]
        return probe.param_table(), [], probe.param_elems, 0

    def _engine(self, N, H, W, training, device):
        pool = self._rt["engines"].setdefault((N, H, W, training), [])
        for e in pool:
            if not e.busy:
                return e
        eng = _DiscriminatorEngine(N, H, W, training, device)
        pool.append(eng)
        return eng

    def last_engine(self):
        return self._rt["last_engine"]

    class _InputGradOnly:
        def __init__(self, module):
            self.m = module

        def __enter__(self):
            self.prev = self.m._rt.get("param_grads", True)
            self.m._rt["param_grads"] = False

        def __exit__(self, *a):
            self.m._rt["param_grads"] = self.prev

    def input_grad_only(self):
        """Context manager: forwards recorded inside back-propagate to the INPUT only (the generator's adversarial
        term, src/train.py:184-190, needs d(D(sr))/d(sr); the reference also fills D's .grad there and then discards
        it with the next d_optimizer.zero_grad())."""
        return Discriminator._InputGradOnly(self)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise RuntimeError("Discriminator (libsrgan_b200) runs on a CUDA device only; there is no CPU path")
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError(f"expected an N x 3 x H x W input, got {tuple(x.shape)}")
        xc = x.contiguous()
        if xc.dtype != torch.float32:
            xc = xc.float()
        N, _, H, W = xc.shape
        self._flatten(xc.device)
        rt = self._rt
        need_grad = torch.is_grad_enabled() and (xc.requires_grad or any(p.requires_grad for p in rt["plist"]))
        eng = self._engine(N, H, W, need_grad, xc.device)
        if need_grad and getattr(eng, "grad_flat", None) is None:
            eng.grad_flat = torch.empty_like(rt["flat"])
        eng.bind(rt["flat"], eng.grad_flat if need_grad else None)
        L = _lib.lib()
        check(L.srg_discriminator_pack(eng.handle, stream_ptr()), "srg_discriminator_pack")
        rt["last_engine"] = eng
        if need_grad:
            _acquire(eng)
            return _DiscriminatorFn.apply(self, eng, xc, *rt["plist"])
        out = torch.empty(N, 512, eng.out_hw[0], eng.out_hw[1], dtype=torch.float32, device=xc.device)
        check(L.srg_discriminator_forward(eng.handle, c_void_p(xc.data_ptr()), c_void_p(out.data_ptr()), stream_ptr()),
              "srg_discriminator_forward")
        return out
