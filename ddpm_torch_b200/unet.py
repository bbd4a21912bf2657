"""Host-side mirror of ``ddpm_torch.models.unet.UNet`` (reference unet.py:92-233) over the sm_100a engine.

Same constructor, same ``state_dict()`` keys / shapes / registration order (so reference checkpoints load with
``load_state_dict`` and EMA / Adam / clip_grad_norm_ / DDP see ordinary ``nn.Parameter``s), same
``forward(x, t)`` contract (x f32[B,C,H,W] NCHW, t i64[B] -> f32[B,C_out,H,W]) — but no ATen graph: the whole
forward and backward run as the engine's launch plan through the C ABI (include/ddpm_b200.h).

All parameters are views into ONE flat fp32 buffer (and gradients come back in one flat buffer), which is what the
kernels read; the bf16 kernel layouts are re-packed from it whenever it changed.  There is no PyTorch/CPU fallback:
calling the model without the built extension or off an sm_100 GPU raises.
"""
import ctypes as C
import math

import torch
import torch.nn as nn

from . import _lib


class _Node(nn.Module):
    """Plain container used only to reproduce the reference's dotted state_dict names."""


def _xavier_uniform_(t, scale):
    """modules.py:11-18 — xavier uniform with gain sqrt(scale or 1e-10)."""
    return nn.init.xavier_uniform_(t, gain=math.sqrt(scale or 1e-10))


class UNet(nn.Module):
    def __init__(self, in_channels, hid_channels, out_channels, ch_multipliers, num_res_blocks, apply_attn,
                 time_embedding_dim=None, drop_rate=0., resample_with_conv=True):
        super().__init__()
        if not resample_with_conv:
            raise NotImplementedError("resample_with_conv=False (AvgPool/plain Upsample) is outside the accelerated path")
        levels = len(ch_multipliers)
        if isinstance(apply_attn, bool):
            apply_attn = [apply_attn] * levels
        self.in_channels, self.hid_channels, self.out_channels = in_channels, hid_channels, out_channels
        self.ch_multipliers, self.apply_attn = tuple(ch_multipliers), tuple(bool(a) for a in apply_attn)
        self.num_res_blocks, self.levels = num_res_blocks, levels
        self.time_embedding_dim = time_embedding_dim or 4 * hid_channels
        self.drop_rate, self.resample_with_conv = drop_rate, resample_with_conv

        cfg = _lib.UnetCfg()
        cfg.in_channels, cfg.hid_channels, cfg.out_channels = in_channels, hid_channels, out_channels
        cfg.levels, cfg.num_res_blocks = levels, num_res_blocks
        for i in range(levels):
            cfg.ch_mult[i] = int(ch_multipliers[i])
            cfg.attn[i] = int(bool(apply_attn[i]))
        cfg.temb_dim, cfg.drop_rate = self.time_embedding_dim, float(drop_rate)
        L = _lib.lib()
        self._cfg = cfg
        self._h = C.c_void_p()
        _lib.check(L.ddpm_unet_create(C.byref(cfg), C.byref(self._h)), "unet_create")
        self._aux = {}                      # auxiliary inference plans (extra handles over the SAME flat parameters)

        # parameter inventory from the engine (reference registration order)
        self._meta = []
        for i in range(L.ddpm_unet_num_params(self._h)):
            name, nd, dims, off = C.c_char_p(), C.c_int(), (C.c_int * 4)(), C.c_longlong()
            _lib.check(L.ddpm_unet_param_info(self._h, i, C.byref(name), C.byref(nd), C.byref(dims), C.byref(off)))
            self._meta.append((name.value.decode(), tuple(dims[:nd.value]), int(off.value)))
        self._flat_elems = int(L.ddpm_unet_flat_elems(self._h))
        flat = torch.zeros(self._flat_elems, dtype=torch.float32)
        self._params = []
        zero_scale = (".conv2.weight", ".project_out.weight", "out_conv.2.weight")   # init_scale=0: unet.py:37,79,141
        for name, shape, off in self._meta:
            n = math.prod(shape)
            p = nn.Parameter(flat[off:off + n].view(shape))
            with torch.no_grad():
                is_norm = ".norm" in name or name.startswith("out_conv.0")
                if name.endswith(".weight") and not is_norm:
                    _xavier_uniform_(p, 0. if name.endswith(zero_scale) else 1.)
                elif name.endswith(".weight"):
                    p.fill_(1.)
            node = self
            *path, leaf = name.split(".")
            for part in path:
                if part not in node._modules:
                    node.add_module(part, _Node())
                node = node._modules[part]
            node.register_parameter(leaf, p)
            self._params.append(p)
        self._flat = flat
        self._grads = None
        self._ws = None
        self._plan_key = None
        self._packed_version = None
        self._packed_epoch = 0
        self._drop_calls = 0
        self._plan_epoch = 0
        self._sampler_cache = {}
        self._acc = None                    # gradient-accumulation buffer (only exists when backward runs twice before a step)
        self._acc_pending = False
        self._bwd_since_zero = 0
        self.register_load_state_dict_post_hook(lambda module, incompatible: module.repack())

    def __del__(self):
        try:
            if getattr(self, "_h", None) is not None and self._h.value:
                _lib.lib().ddpm_unet_destroy(self._h)
                self._h = C.c_void_p()
            for a in getattr(self, "_aux", {}).values():
                _lib.lib().ddpm_unet_destroy(a["h"])
            self._aux = {}
        except Exception:
            pass

    # ------------------------------------------------------------------ flat-buffer maintenance
    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)     # .to()/.cuda()/.float() give every parameter its own storage ...
        self._reflatten()                     # ... so gather them back into one flat buffer
        return out

    def _reflatten(self):
        dev = self._params[0].device
        flat = torch.zeros(self._flat_elems, dtype=torch.float32, device=dev)
        with torch.no_grad():
            for p, (_, shape, off) in zip(self._params, self._meta):
                n = p.numel()
                flat[off:off + n].copy_(p.detach().reshape(-1).to(torch.float32))
                p.data = flat[off:off + n].view(shape)
        self._flat = flat
        self._plan_key = None
        self._packed_version = None
        self._sampler_cache = {}

    def _views_ok(self):
        base = self._flat.data_ptr()
        return all(p.data_ptr() == base + 4 * off for p, (_, _, off) in zip(self._params, self._meta))

    @property
    def flat_params(self):
        return self._flat

    @property
    def flat_grads(self):
        """Flat fp32 gradient buffer = SUM of the backward passes since the last ``zero_grad`` / optimizer step (the
        reference accumulates in ``p.grad`` with ``--num-accum``, train.py / utils/train.py:152-165).  The engine's backward
        overwrites its buffer, so earlier micro-batches are parked in ``_acc`` and folded back in here."""
        if self._acc_pending:
            self._grads.add_(self._acc)
            self._acc_pending = False
        return self._grads

    def _before_backward(self):
        if self._bwd_since_zero > 0:        # a previous micro-batch's gradient is still unconsumed: park it
            g = self.flat_grads
            if self._acc is None or self._acc.device != g.device:
                self._acc = torch.empty_like(g)
            self._acc.copy_(g)
            self._acc_pending = True
        self._bwd_since_zero += 1

    def grads_consumed(self):
        """Called by ``FusedAdam.step`` / ``zero_grad``: the next backward starts a fresh accumulation."""
        self._bwd_since_zero = 0
        self._acc_pending = False

    def zero_grad(self, set_to_none=True):
        self.grads_consumed()
        return super().zero_grad(set_to_none)

    def _weights_version(self):
        """Changes whenever a parameter was written through autograd-visible ops: optimizer steps, ``load_state_dict``,
        ``p.copy_``.  After ``.cuda()`` the parameters no longer share the flat buffer's version counter (``p.data = view``),
        so the per-parameter counters are summed.  ``p.data.copy_`` (the reference EMA swap, utils/train.py:307-316) bumps
        NO counter: the sampler loops therefore re-pack unconditionally at their head (0.2 ms per loop)."""
        return (self._flat._version, sum(p._version for p in self._params), self._packed_epoch)

    def grad_views(self, flat=None):
        flat = self._grads if flat is None else flat
        return [flat[off:off + math.prod(shape)].view(shape) for _, shape, off in self._meta]

    # ------------------------------------------------------------------ planning
    def prepare(self, B, H, W, training, force_repack=False):
        """Compile (or reuse) the launch plan for this batch shape and (re)pack weights if they changed."""
        if not self._flat.is_cuda:
            raise RuntimeError("ddpm_torch_b200.UNet runs on sm_100a CUDA devices only (no CPU / PyTorch fallback); "
                               "move the model with .cuda() first")
        if not self._views_ok():
            self._reflatten()
        L = _lib.lib()
        key = (B, H, W, bool(training), self._flat.data_ptr())
        if key != self._plan_key:
            need = L.ddpm_unet_workspace_bytes(self._h, B, H, W, int(training))
            if need < 0:
                _lib.check(int(need), "workspace_bytes")
            dev = self._flat.device
            if self._ws is None or self._ws.numel() < need or self._ws.device != dev:
                if self._ws is not None:
                    torch.cuda.synchronize(self._ws.device)     # the engine's side stream may still hold a queued weight re-pack into it
                self._ws = None
                self._ws = torch.empty(int(need), dtype=torch.uint8, device=dev)
            if training and (self._grads is None or self._grads.device != dev):
                self._grads = torch.zeros(self._flat_elems, dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                _lib.check(L.ddpm_unet_plan(self._h, B, H, W, int(training), self._flat.data_ptr(),
                                            self._grads.data_ptr() if training else None,
                                            self._ws.data_ptr(), self._ws.numel()), "unet_plan")
            self._plan_key = key
            self._plan_epoch += 1                 # captured sampler graphs of older plans are stale (see diffusion._native_sample_loop)
            self._packed_version = None
        self.repack_if_needed(force=training or force_repack)
        return self._h

    def aux_plan(self, idx, B, H, W, force=False):
        """Extra inference plan #idx over the same flat parameters with its own workspace (the sampler runs two half
        batches on two streams so that one half's HBM-bound GroupNorm kernels overlap the other's tensor-core kernels).
        Returns the handle; its packed weights are refreshed whenever the parameters changed."""
        if not self._flat.is_cuda:
            raise RuntimeError("ddpm_torch_b200.UNet runs on sm_100a CUDA devices only (no CPU / PyTorch fallback)")
        if not self._views_ok():
            self._reflatten()
        L = _lib.lib()
        a = self._aux.get(idx)
        key = (B, H, W, self._flat.data_ptr())
        if a is None or a["key"] != key:
            if a is None:
                h = C.c_void_p()
                _lib.check(L.ddpm_unet_create(C.byref(self._cfg), C.byref(h)), "unet_create")
                a = {"h": h, "ws": None, "key": None, "ver": None}
                self._aux[idx] = a
            need = L.ddpm_unet_workspace_bytes(a["h"], B, H, W, 0)
            if need < 0:
                _lib.check(int(need), "workspace_bytes")
            if a["ws"] is None or a["ws"].numel() < need or a["ws"].device != self._flat.device:
                a["ws"] = None
                a["ws"] = torch.empty(int(need), dtype=torch.uint8, device=self._flat.device)
            with torch.cuda.device(self._flat.device):
                _lib.check(L.ddpm_unet_plan(a["h"], B, H, W, 0, self._flat.data_ptr(), None, a["ws"].data_ptr(), a["ws"].numel()), "unet_plan")
            a["key"], a["ver"] = key, None
            a["epoch"] = a.get("epoch", 0) + 1
        if force or a["ver"] != self._weights_version():
            with torch.cuda.device(self._flat.device):
                _lib.check(L.ddpm_unet_repack(a["h"], _lib.stream_ptr(self._flat.device)), "unet_repack")
            a["ver"] = self._weights_version()
        return a["h"]

    def repack_if_needed(self, force=False):
        v = self._weights_version()
        if force or v != self._packed_version:
            with torch.cuda.device(self._flat.device):
                _lib.check(_lib.lib().ddpm_unet_repack(self._h, _lib.stream_ptr(self._flat.device)), "unet_repack")
            self._packed_version = v

    def repack(self):
        """Call after out-of-band weight edits (e.g. ``p.data.copy_`` as the reference EMA does, utils/train.py:307-316)."""
        self._packed_version = None
        self._packed_epoch += 1

    def next_dropout_seed(self):
        self._drop_calls += 1
        return (torch.initial_seed() * 1000003 + self._drop_calls) & 0xFFFFFFFFFFFFFFFF

    # ------------------------------------------------------------------ forward
    def forward(self, x, t):
        B, Cc, H, W = x.shape
        assert Cc == self.in_channels
        x = x.contiguous().float()
        t = t.contiguous().to(torch.int64)
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self._params)
        if need_grad:
            return _UNetFn.apply(self, x, t, *self._params)
        return self._forward_nograd(x, t)

    def _forward_nograd(self, x, t, training_plan=False):
        B, _, H, W = x.shape
        h = self.prepare(B, H, W, training_plan)
        out = torch.empty(B, self.out_channels, H, W, dtype=torch.float32, device=x.device)
        seed = self.next_dropout_seed() if (self.training and self.drop_rate > 0) else 0
        dev = self._flat.device
        if x.device != dev or t.device != dev:
            raise RuntimeError(f"UNet lives on {dev} but got x on {x.device}, t on {t.device}")
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ddpm_unet_forward(h, x.data_ptr(), t.data_ptr(), out.data_ptr(), seed, _lib.stream_ptr(dev)),
                       "unet_forward")
        return out


class _UNetFn(torch.autograd.Function):
    """Autograd bridge: parameter gradients come back as views of one freshly cloned flat buffer."""

    @staticmethod
    def forward(ctx, model, x, t, *params):
        out = model._forward_nograd(x, t, training_plan=True)
        ctx.model = model
        ctx.save_for_backward(x, t)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        model = ctx.model
        g = grad_out.contiguous().float()
        dev = model._flat.device
        model._before_backward()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ddpm_unet_backward(model._h, g.data_ptr(), _lib.stream_ptr(dev)), "unet_backward")
        flat = model._grads.clone()
        return (None, None, None, *model.grad_views(flat))


class ModelWrapper(nn.Module):
    """utils/train.py:349-367: optional pre / post transforms around a model (the reference uses PixelUnshuffle / PixelShuffle
    when ``block_size > 1``, train.py:70-73).  ``ModelWrapper(UNet(C*b*b, ...), nn.PixelUnshuffle(b), nn.PixelShuffle(b))`` (also
    inside DDP) takes the diffusion classes' native training and sampling paths on the unshuffled layout; with any other
    transforms the wrapper is a generic ``denoise_fn`` (torch formulas, the inner ``UNet`` still executes on the engine)."""

    def __init__(self, model, pre_transform=None, post_transform=None):
        super().__init__()
        self._model = model
        self.pre_transform = pre_transform
        self.post_transform = post_transform

    def forward(self, x, *args, **kwargs):
        if self.pre_transform is not None:
            x = self.pre_transform(x)
        out = self._model(x, *args, **kwargs)
        return out if self.post_transform is None else self.post_transform(out)
