"""Host-side mirror of ``ddpm_torch.diffusion`` (reference diffusion.py) for the accelerated path.

``GaussianDiffusion`` keeps the reference's constructor, attribute names (fp64 coefficient tables) and method
signatures.  When ``denoise_fn`` is a ``ddpm_torch_b200.UNet`` (optionally wrapped in DDP / a ``.module`` holder) and
the configuration is the one every reference config uses (eps-prediction, fixed variance, mse loss):

* ``train_losses``  -> one fused engine call: q_sample prologue, UNet forward, per-sample MSE (and the matching
  fused backward through autograd),
* ``p_sample`` / ``p_sample_step`` -> the engine's sampler step (UNet forward + the alpha/beta update of
  diffusion.py:107-158 in one launch sequence, replayed from a CUDA graph once per timestep).

A block-size model (train.py:63-73: ``ModelWrapper(UNet(C*b*b, ...), PixelUnshuffle(b), PixelShuffle(b))``, optionally inside
DDP) takes the same native paths on the inner layout [B, C*b*b, H/b, W/b]; the pixel (un)shuffles are torch copies around them.
Any other ``denoise_fn`` (toy MLPs, other wrappers) takes the generic formulas below, written with plain torch ops.
"""
import ctypes as C

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .unet import UNet


def get_beta_schedule(beta_schedule, beta_start, beta_end, timesteps, dtype=torch.float64):
    """Same schedules and fp64 arithmetic as diffusion.py:13-29."""
    lin = lambda a, b, n: torch.linspace(a, b, n, dtype=dtype)
    if beta_schedule == "linear":
        betas = lin(beta_start, beta_end, timesteps)
    elif beta_schedule == "quad":
        betas = lin(beta_start ** 0.5, beta_end ** 0.5, timesteps) ** 2
    elif beta_schedule in ("warmup10", "warmup50"):
        n = int(timesteps * (0.1 if beta_schedule == "warmup10" else 0.5))
        betas = torch.full((timesteps,), beta_end, dtype=dtype)
        betas[:n] = lin(beta_start, beta_end, n)
    elif beta_schedule == "const":
        betas = torch.full((timesteps,), beta_end, dtype=dtype)
    elif beta_schedule == "jsd":
        betas = 1. / lin(timesteps, 1, timesteps)
    else:
        raise NotImplementedError(beta_schedule)
    assert betas.shape == (timesteps,)
    return betas


def _native(denoise_fn):
    """Unwrap DDP / holders and a pixel (un)shuffle model wrapper (utils/train.py:349-367); return (engine UNet, block size b)
    or (None, 1).  A wrapper counts only when its transforms are exactly PixelUnshuffle(b) / PixelShuffle(b) with the same b
    around an engine UNet: the native paths then run the UNet on pixel_unshuffle(x, b) and shuffle its output back."""
    m = denoise_fn
    for _ in range(3):
        if isinstance(m, UNet):
            return m, 1
        pre, post = getattr(m, "pre_transform", None), getattr(m, "post_transform", None)
        if hasattr(m, "_model") and type(pre) is nn.PixelUnshuffle and type(post) is nn.PixelShuffle:
            inner = m._model
            if pre.downscale_factor == post.upscale_factor and isinstance(inner, UNet):
                return inner, pre.downscale_factor
            return None, 1
        m = getattr(m, "module", None)
        if m is None:
            return None, 1
    return None, 1


def _to_inner(x, model, b):
    """pixel_unshuffle(x, b) as a contiguous fp32 batch for the engine UNet of a block-size model, whose plan reads exactly
    model.in_channels channels."""
    if x.shape[1] * b * b != model.in_channels:
        raise ValueError(f"block size {b}: the UNet takes {model.in_channels} channels, the batch has {x.shape[1]}")
    return F.pixel_unshuffle(x.float(), b).contiguous()


def _unshuffle_into(dst, src, b):
    """dst[B, C*b*b, H/b, W/b] = pixel_unshuffle(src[B, C, H, W], b) as one copy into an existing buffer (no allocation, so it can
    sit inside a captured graph)."""
    B, Cc, H, W = src.shape
    dst.view(B, Cc, b, b, H // b, W // b).copy_(src.view(B, Cc, H // b, b, W // b, b).permute(0, 1, 3, 5, 2, 4))


def _flat_mean(x):
    return x.mean(dim=list(range(1, x.ndim)))


def _coef_tables(betas=None, alphas_bar=None, eta2=None):
    """All fp64 coefficient tables as a dict keyed by the reference's attribute names.

    ``betas`` given: the full-chain tables of diffusion.py:52-67.  ``alphas_bar`` given (already restricted to a
    sub-sequence) with ``eta2 = eta**2``: the DDIM re-derivation of ddim.py:61-92.  Every expression keeps the reference's
    operand order, so the tables are bit-identical (tests/test_oracle_golden.py::test_mirror_tables_bit_exact)."""
    T = {}
    one = torch.ones(1, dtype=torch.float64)
    if alphas_bar is None:
        alphas = 1 - betas
        ab = torch.cumprod(alphas, dim=0)
        prev = torch.cat([one, ab[:-1]])
    else:
        ab = alphas_bar
        prev = torch.cat([one, ab[:-1]], dim=0)
        alphas = ab / prev
        betas = 1. - alphas
        T.update(betas=betas, alphas=alphas, alphas_bar_prev=prev, sqrt_alphas_bar_prev=prev.sqrt())
    rest = 1. - ab                                     # 1 - alpha_bar_t
    T.update(alphas_bar=ab, sqrt_alphas_bar=ab.sqrt(), sqrt_one_minus_alphas_bar=rest.sqrt(),
             sqrt_recip_alphas_bar=(1. / ab).sqrt(), sqrt_recip_m1_alphas_bar=(1. / ab - 1.).sqrt())
    if eta2 is None:
        pv = betas * (1. - prev) / rest
        T.update(posterior_var=pv, posterior_logvar_clipped=torch.log(torch.cat([pv[[1]], pv[1:]])),
                 posterior_mean_coef1=betas * prev.sqrt() / rest, posterior_mean_coef2=alphas.sqrt() * (1. - prev) / rest)
    else:
        pv = betas * (1. - prev) / rest * eta2
        c2 = (1 - ab - eta2 * betas).sqrt() * (1 - prev).sqrt() / rest
        T.update(posterior_var=pv, posterior_logvar_clipped=torch.log(torch.cat([pv[[1]], pv[1:]]).clip(min=1e-20)),
                 posterior_mean_coef2=c2, posterior_mean_coef1=prev.sqrt() * (1. - alphas.sqrt() * c2))
    return T


class GaussianDiffusion:
    def __init__(self, betas, model_mean_type, model_var_type, loss_type, **kwargs):
        assert isinstance(betas, torch.Tensor) and betas.dtype == torch.float64
        assert (betas > 0).all() and (betas <= 1).all()
        self.betas = betas
        self.model_mean_type, self.model_var_type, self.loss_type = model_mean_type, model_var_type, loss_type
        self.timesteps = len(betas)
        self.__dict__.update(_coef_tables(betas))
        self._set_fixed_var(clip=False)
        self._dev_cache = {}

    def _set_fixed_var(self, clip):
        large = torch.cat([self.posterior_var[[1]], self.betas[1:]])
        if clip:
            large = large.clip(min=1e-20)
        self.fixed_model_var, self.fixed_model_logvar = {
            "fixed-large": (self.betas, torch.log(large)),
            "fixed-small": (self.posterior_var, self.posterior_logvar_clipped),
        }.get(self.model_var_type, (None, None))

    # ------------------------------------------------------------------ generic (torch) formulas
    @staticmethod
    def _extract(arr, t, x, dtype=torch.float32, device=torch.device("cpu"), ndim=4):
        if x is not None:
            dtype, device, ndim = x.dtype, x.device, x.ndim
        out = torch.as_tensor(arr, dtype=dtype, device=device).gather(0, t)
        return out.reshape((-1,) + (1,) * (ndim - 1))

    def q_mean_var(self, x_0, t):
        return (self._extract(self.sqrt_alphas_bar, t, x_0) * x_0, self._extract(1. - self.alphas_bar, t, x_0),
                self._extract(torch.log(1 - self.alphas_bar), t, x_0))

    def q_sample(self, x_0, t, noise=None):
        if noise is None:
            noise = torch.randn_like(x_0)
        return self._extract(self.sqrt_alphas_bar, t, x_0) * x_0 + \
            self._extract(self.sqrt_one_minus_alphas_bar, t, x_0) * noise

    def q_posterior_mean_var(self, x_0, x_t, t):
        mean = self._extract(self.posterior_mean_coef1, t, x_0) * x_0 + self._extract(self.posterior_mean_coef2, t, x_0) * x_t
        return mean, self._extract(self.posterior_var, t, x_0), self._extract(self.posterior_logvar_clipped, t, x_0)

    def _pred_x_0_from_eps(self, x_t, eps, t):
        return self._extract(self.sqrt_recip_alphas_bar, t, x_t) * x_t - self._extract(self.sqrt_recip_m1_alphas_bar, t, x_t) * eps

    def _pred_x_0_from_mean(self, x_t, mean, t):
        c1, c2 = self._extract(self.posterior_mean_coef1, t, x_t), self._extract(self.posterior_mean_coef2, t, x_t)
        return mean / c1 - c2 / c1 * x_t

    def p_mean_var(self, denoise_fn, x_t, t, clip_denoised, return_pred):
        out = denoise_fn(x_t, t)
        if self.model_var_type == "learned":
            out, model_logvar = out.chunk(2, dim=1)
            model_var = torch.exp(model_logvar)
        elif self.model_var_type in ("fixed-small", "fixed-large"):
            model_var, model_logvar = self._extract(self.fixed_model_var, t, x_t), self._extract(self.fixed_model_logvar, t, x_t)
        else:
            raise NotImplementedError(self.model_var_type)
        clip = (lambda v: v.clamp(-1., 1.)) if clip_denoised else (lambda v: v)
        if self.model_mean_type == "mean":
            pred_x_0, model_mean = clip(self._pred_x_0_from_mean(x_t, out, t)), out
        elif self.model_mean_type == "x_0":
            pred_x_0 = clip(out)
            model_mean = self.q_posterior_mean_var(pred_x_0, x_t, t)[0]
        elif self.model_mean_type == "eps":
            pred_x_0 = clip(self._pred_x_0_from_eps(x_t, out, t))
            model_mean = self.q_posterior_mean_var(pred_x_0, x_t, t)[0]
        else:
            raise NotImplementedError(self.model_mean_type)
        return (model_mean, model_var, model_logvar, pred_x_0) if return_pred else (model_mean, model_var, model_logvar)

    def _fast_ok(self, denoise_fn):
        """(engine UNet, block size) when the native paths apply, else (None, 1)."""
        m, b = _native(denoise_fn)
        ok = m is not None and self.model_mean_type == "eps" and self.model_var_type in ("fixed-small", "fixed-large")
        return (m, b) if ok else (None, 1)

    # ------------------------------------------------------------------ sampling
    def p_sample_step(self, denoise_fn, x_t, t, clip_denoised=True, return_pred=False, generator=None):
        model_mean, _, model_logvar, pred_x_0 = self.p_mean_var(denoise_fn, x_t, t, clip_denoised, True)
        noise = torch.empty_like(x_t).normal_(generator=generator)
        nonzero = (t > 0).reshape((-1,) + (1,) * (x_t.ndim - 1)).to(x_t)
        sample = model_mean + nonzero * torch.exp(0.5 * model_logvar) * noise
        return (sample, pred_x_0) if return_pred else sample

    def _coef_rows(self):
        """[S,6] fp32 rows {sqrt_recip_ab, sqrt_recip_m1_ab, c1, c2, exp(.5*logvar), t>0}; every entry goes through the
        same fp64 -> fp32 cast as ``_extract`` (diffusion.py:83) and sigma is exp(0.5*fp32(logvar)) as in :157."""
        f = lambda a: torch.as_tensor(a, dtype=torch.float32)
        S = len(self.betas)
        nz = (torch.arange(S) > 0).float()
        return torch.stack([f(self.sqrt_recip_alphas_bar), f(self.sqrt_recip_m1_alphas_bar), f(self.posterior_mean_coef1),
                            f(self.posterior_mean_coef2), torch.exp(0.5 * f(self.fixed_model_logvar)), nz], dim=1).contiguous()

    def _model_timesteps(self):
        return torch.arange(len(self.betas), dtype=torch.int64)

    @torch.inference_mode()
    def p_sample(self, denoise_fn, shape=None, device=torch.device("cpu"), noise=None, seed=None, rng="torch", use_graph=True, split=None):
        """diffusion.py:160-174.  ``rng="torch"`` consumes a torch.Generator exactly like the reference (bit-identical
        noise stream); ``rng="philox"`` draws the per-step noise inside the step kernel (one launch sequence per step)."""
        model, blk = self._fast_ok(denoise_fn)
        B = (shape or noise.shape)[0]
        gen = torch.Generator(device).manual_seed(seed) if seed is not None else None
        x_t = torch.empty(shape, device=device).normal_(generator=gen) if noise is None else noise.to(device)
        S = len(self.betas)
        if model is None:
            t = torch.empty((B,), dtype=torch.int64, device=device)
            fn = self._wrap_denoise(denoise_fn, device)
            for ti in range(S - 1, -1, -1):
                t.fill_(ti)
                x_t = self.p_sample_step(fn, x_t, t, generator=gen)
            return x_t
        if blk > 1:        # x_T is drawn in the outer shape, as the reference does, and the chain runs on the UNet's layout
            return F.pixel_shuffle(_native_sample_loop(self, model, _to_inner(x_t, model, blk), gen, rng, seed, use_graph, split, blk), blk)
        return _native_sample_loop(self, model, x_t.contiguous().float().clone(), gen, rng, seed, use_graph, split)

    def _wrap_denoise(self, denoise_fn, device):
        return denoise_fn

    @torch.inference_mode()
    def p_sample_progressive(self, denoise_fn, shape, device=torch.device("cpu"), noise=None, pred_freq=10, seed=None):
        """diffusion.py:176-198.  Native path: every step is the engine's sampler step, which also writes the clipped x_0
        prediction (ddpm_sampler_step_pred); predictions are copied out every ``pred_freq`` steps exactly as the reference does."""
        B = (shape or noise.shape)[0]
        gen = torch.Generator(device).manual_seed(seed) if seed is not None else None
        x_t = torch.empty(shape, device=device).normal_(generator=gen) if noise is None else noise.to(device)
        n = self.timesteps // pred_freq
        preds = torch.zeros((n, B) + tuple(shape[1:]), dtype=torch.float32)
        idx = n
        model, blk = self._fast_ok(denoise_fn)
        if model is not None and x_t.is_cuda:
            L = _lib.lib()
            dev = model.flat_params.device
            x_out = x_t
            x_t = _to_inner(x_t, model, blk) if blk > 1 else x_t.contiguous().float().clone()
            _, _, H, W = x_t.shape
            was_training = model.training
            model.eval()
            try:
                with torch.cuda.device(dev):
                    h = model.prepare(B, H, W, training=False, force_repack=True)
                    coef, tmod = self._coef_rows(), self._model_timesteps().contiguous()
                    _lib.check(L.ddpm_sampler_setup(h, coef.shape[0], tmod.data_ptr(), coef.data_ptr()), "sampler_setup")
                    _lib.check(L.ddpm_sampler_reset(h, self.timesteps - 1, _lib.stream_ptr(dev)), "sampler_reset")
                    z, pred = torch.empty_like(x_t), torch.empty_like(x_t)
                    z_out = torch.empty_like(x_out) if blk > 1 else z      # noise is drawn in the outer shape (diffusion.py:155)
                    for ti in range(self.timesteps - 1, -1, -1):
                        z_out.normal_(generator=gen)
                        if blk > 1:
                            _unshuffle_into(z, z_out, blk)
                        _lib.check(L.ddpm_sampler_step_pred(h, x_t.data_ptr(), z.data_ptr(), 0, pred.data_ptr(), _lib.stream_ptr(dev)), "sampler_step")
                        if (ti + 1) % pred_freq == 0:
                            idx -= 1
                            preds[idx] = (F.pixel_shuffle(pred, blk) if blk > 1 else pred).cpu()
            finally:
                if was_training:
                    model.train()
            return (F.pixel_shuffle(x_t, blk) if blk > 1 else x_t).cpu(), preds
        t = torch.empty(B, dtype=torch.int64, device=device)
        fn = self._wrap_denoise(denoise_fn, device)
        for ti in range(self.timesteps - 1, -1, -1):
            t.fill_(ti)
            x_t, pred = self.p_sample_step(fn, x_t, t, return_pred=True, generator=gen)
            if (ti + 1) % pred_freq == 0:
                idx -= 1
                preds[idx] = pred.cpu()
        return x_t.cpu(), preds

    # ------------------------------------------------------------------ training
    def train_losses(self, denoise_fn, x_0, t, noise=None):
        if noise is None:
            noise = torch.randn_like(x_0)
        model, blk = self._fast_ok(denoise_fn)
        if model is not None and self.loss_type == "mse" and x_0.is_cuda:
            if blk > 1:
                # q_sample is elementwise and the per-sample mean is invariant under the pixel permutation: the fused loss on the
                # unshuffled batch is the reference's loss of the wrapped model
                x_0, noise = _to_inner(x_0, model, blk), _to_inner(noise, model, blk)
            return _TrainLossFn.apply(self, model, denoise_fn, x_0.contiguous().float(), t.contiguous(), noise.contiguous().float(),
                                      *model._params)
        x_t = self.q_sample(x_0, t, noise=noise)
        if self.loss_type == "kl":      # diffusion.py:226-228: weighted variational bound, generic torch path only
            return self._loss_term_bpd(denoise_fn, x_0=x_0, x_t=x_t, t=t, clip_denoised=False, return_pred=False)
        if self.loss_type != "mse":
            raise NotImplementedError(self.loss_type)
        assert self.model_var_type != "learned"
        target = {"mean": lambda: self.q_posterior_mean_var(x_0, x_t, t)[0], "x_0": lambda: x_0, "eps": lambda: noise}[self.model_mean_type]()
        return _flat_mean((target - denoise_fn(x_t, t)).pow(2))

    # ------------------------------------------------------------------ log-likelihood in bits per dimension (generic torch)
    def _loss_term_bpd(self, denoise_fn, x_0, x_t, t, clip_denoised, return_pred):
        """diffusion.py:203-215: L_t = KL(q(x_{t-1}|x_t,x_0) || p(x_{t-1}|x_t)) for t > 0, decoder NLL -log p(x_0|x_1) at t = 0."""
        from .functions import discretized_gaussian_loglik, flat_mean, normal_kl
        true_mean, _, true_logvar = self.q_posterior_mean_var(x_0=x_0, x_t=x_t, t=t)
        model_mean, _, model_logvar, pred_x_0 = self.p_mean_var(denoise_fn, x_t=x_t, t=t, clip_denoised=clip_denoised, return_pred=True)
        kl = flat_mean(normal_kl(true_mean, true_logvar, model_mean, model_logvar)) / math.log(2.)
        nll = flat_mean(-discretized_gaussian_loglik(x_0, model_mean, log_scale=0.5 * model_logvar)) / math.log(2.)
        out = torch.where(t.to(kl.device) > 0, kl, nll)
        return (out, pred_x_0) if return_pred else out

    def _prior_bpd(self, x_0):
        """diffusion.py:245-250: KL(q(x_T|x_0) || N(0, I)) in bits per dimension."""
        from .functions import flat_mean, normal_kl
        B, T = len(x_0), self.timesteps
        T_mean, _, T_logvar = self.q_mean_var(x_0=x_0, t=(T - 1) * torch.ones((B,), dtype=torch.int64))
        zero = torch.zeros((), dtype=T_mean.dtype, device=T_mean.device)
        return flat_mean(normal_kl(T_mean, T_logvar, zero, zero)) / math.log(2.)

    def calc_all_bpd(self, denoise_fn, x_0, clip_denoised=True):
        """diffusion.py:252-270.  Upstream unpacks ``B, T = x_0.shape, self.timesteps`` (B becomes the shape tuple and
        ``torch.empty([B, ])`` raises, SURVEY §2 row 4); this is the evident intent, B = batch size.
        Returns (total_bpd [B], losses [B, T], prior_bpd [B], mses [B, T])."""
        from .functions import flat_mean
        B, T = len(x_0), self.timesteps
        t = torch.empty([B, ], dtype=torch.int64)
        losses = torch.zeros([B, T], dtype=torch.float32)
        mses = torch.zeros([B, T], dtype=torch.float32)
        for ti in range(T - 1, -1, -1):
            t.fill_(ti)
            x_t = self.q_sample(x_0, t=t)
            loss, pred_x_0 = self._loss_term_bpd(denoise_fn, x_0, x_t=x_t, t=t, clip_denoised=clip_denoised, return_pred=True)
            losses[:, ti] = loss
            mses[:, ti] = flat_mean((pred_x_0 - x_0).pow(2))
        prior_bpd = self._prior_bpd(x_0)
        total_bpd = torch.sum(losses, dim=1) + prior_bpd
        return total_bpd, losses, prior_bpd, mses

    def _dev_tables(self, device):
        k = str(device)
        if k not in self._dev_cache:
            self._dev_cache[k] = (torch.as_tensor(self.sqrt_alphas_bar, dtype=torch.float32, device=device).contiguous(),
                                  torch.as_tensor(self.sqrt_one_minus_alphas_bar, dtype=torch.float32, device=device).contiguous())
        return self._dev_cache[k]


class _TrainLossFn(torch.autograd.Function):
    """losses[b] = mean((noise - UNet(q_sample(x0,t,noise), t))^2) through ddpm_train_forward / ddpm_train_backward."""

    @staticmethod
    def forward(ctx, diffusion, model, wrapper, x0, t, noise, *params):
        B, _, H, W = x0.shape
        train = torch.is_grad_enabled() or any(p.requires_grad for p in params)
        dev = model.flat_params.device
        if x0.device != dev:
            raise RuntimeError(f"UNet lives on {dev} but the batch is on {x0.device}")
        h = model.prepare(B, H, W, training=train)
        ta, ts = diffusion._dev_tables(dev)
        losses = torch.empty(B, dtype=torch.float32, device=dev)
        seed = model.next_dropout_seed() if (model.training and model.drop_rate > 0) else 0
        t = t.to(device=dev, dtype=torch.int64)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ddpm_train_forward(h, x0.data_ptr(), t.data_ptr(), noise.data_ptr(), ta.data_ptr(), ts.data_ptr(),
                                                     losses.data_ptr(), seed, _lib.stream_ptr(dev)), "train_forward")
        ctx.model = model
        ctx.wrapper = wrapper
        ctx.keep = (x0, t, noise)
        return losses

    @staticmethod
    def backward(ctx, g):
        model = ctx.model
        g = g.contiguous().float()
        dev = model.flat_params.device
        model._before_backward()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().ddpm_train_backward(model._h, g.data_ptr(), _lib.stream_ptr(dev)), "train_backward")
        _ddp_allreduce(ctx.wrapper, model)
        flat = model._grads.clone()
        return (None, None, None, None, None, None, *model.grad_views(flat))


def _ddp_allreduce(wrapper, model):
    """The fused path calls the inner UNet directly, so a DistributedDataParallel wrapper's ``forward`` never runs and its
    reducer stays disarmed (its autograd hooks return early) - the replicas would silently diverge under the reference flow
    ``DDP(model)`` + ``diffusion.train_losses(self.model, ...)`` (train.py:110, utils/train.py:144-153).  The engine owns the
    collective instead: ONE mean all-reduce of the flat gradient buffer over the wrapper's process group, issued here,
    before autograd hands the views to ``p.grad``.  (If the reducer happens to be armed, averaging already-equal
    gradients again is the identity.)"""
    import torch.distributed as dist
    if wrapper is model or not (dist.is_available() and dist.is_initialized()):
        return
    if not hasattr(wrapper, "process_group") and not hasattr(wrapper, "module"):
        return
    from .parallel import allreduce_grads_overlapped_
    allreduce_grads_overlapped_(model, group=getattr(wrapper, "process_group", None))     # chunk-wise, overlapped with the backward's tail


def _native_sample_loop(diffusion, model, x, gen, rng, seed, use_graph, split=None, blk=1):
    """T sampler steps on the engine: per step {noise draw, step-table fetch, UNet forward with the alpha/beta update in the final
    conv's epilogue}; captured once, replayed T times - one graph launch per timestep.

    ``blk > 1`` (block-size model): ``x`` is already in the UNet's layout [B, C*b*b, H/b, W/b]; each step's torch noise is drawn in
    the outer shape [B, C, H, W] and unshuffled into the step's noise buffer, so the stream is the reference's draw for draw.

    ``split=2`` (opt-in; DDPM_SAMPLER_SPLIT overrides the default of 1 - measured on B200 at bs=256: 5.46 vs 5.47 ms per step, no gain, since half-batch kernels are less efficient): the batch is cut into two
    halves with their own plans, run on two forked streams inside the SAME captured graph, so that one half's HBM-bound
    GroupNorm kernels overlap the other half's tensor-core kernels.  Images and noise are per-sample, so the result is
    the same as the unsplit loop."""
    import os
    L = _lib.lib()
    B, _, H, W = x.shape
    was_training = model.training
    model.eval()
    if split is None:
        split = int(os.environ.get("DDPM_SAMPLER_SPLIT", "1"))
    if split not in (1, 2) or B % split:
        raise ValueError("sampler split must be 1 or 2 and divide the batch")
    Bh = B // split
    dev = model.flat_params.device
    if x.device != dev:
        raise RuntimeError(f"UNet lives on {dev} but the sampler state is on {x.device}")
    ctx_dev = torch.cuda.device(dev)
    ctx_dev.__enter__()          # every launch below targets the model's device (generate.py:59 never calls set_device)
    try:
        return _native_sample_loop_on_device(diffusion, model, x, gen, rng, seed, use_graph, split, Bh, H, W, was_training, blk)
    finally:
        ctx_dev.__exit__(None, None, None)
        if was_training:
            model.train()


def _native_sample_loop_on_device(diffusion, model, x, gen, rng, seed, use_graph, split, Bh, H, W, was_training, blk=1):
    L = _lib.lib()
    # weights are re-packed unconditionally at the head of every loop: the reference EMA swaps values with `p.data.copy_`
    # (utils/train.py:307-316), which no version counter sees; 0.2 ms against a T-step loop
    hs = [model.prepare(Bh, H, W, training=False, force_repack=True)] + [model.aux_plan(i, Bh, H, W, force=True) for i in range(1, split)]
    coef = diffusion._coef_rows()
    tmod = diffusion._model_timesteps().contiguous()
    S = coef.shape[0]
    pseed = 0 if rng == "torch" else ((seed if seed is not None else torch.initial_seed()) | 1) & 0xFFFFFFFFFFFFFFFF
    # The captured step graph is CACHED on the model per (plan, batch shape, chain length, generator kind): generate.py calls
    # p_sample once per batch, and re-capturing ~150 kernels per call costs more than a dozen DDIM steps.  A cached graph owns
    # persistent x / z buffers and (for seeded runs) a persistent registered generator that takes over the caller's generator state.
    ent = None
    B, Cc = x.shape[:2]
    outer = (B, Cc // (blk * blk), H * blk, W * blk)
    if use_graph and rng == "torch" and S > 1:
        key = (x.shape, blk, split, S, gen is not None, model._plan_epoch, tuple(model._aux[i].get("epoch", 0) for i in range(1, split)))
        ent = model._sampler_cache.get(key)
        if ent is None:
            if len(model._sampler_cache) >= 4:
                model._sampler_cache.clear()
            ent = model._sampler_cache[key] = {"x": torch.empty_like(x), "z": torch.empty_like(x), "graph": None,
                                               "z_out": x.new_empty(outer) if blk > 1 else None,
                                               "gen": torch.Generator(x.device) if gen is not None else None}
        xb, z, z_out = ent["x"], ent["z"], ent["z_out"]
        xb.copy_(x)
        x = xb
        if gen is not None:
            ent["gen"].set_state(gen.get_state())      # continue the caller's stream (x_T may already have been drawn from it)
            gen = ent["gen"]
    else:
        z = torch.empty_like(x) if rng == "torch" else None
        z_out = x.new_empty(outer) if (rng == "torch" and blk > 1) else None
    stream = torch.cuda.current_stream()
    for h in hs:
        _lib.check(L.ddpm_sampler_setup(h, S, tmod.data_ptr(), coef.data_ptr()), "sampler_setup")
        _lib.check(L.ddpm_sampler_reset(h, S - 1, C.c_void_p(stream.cuda_stream)), "sampler_reset")
    xs = [x[i * Bh:(i + 1) * Bh] for i in range(split)]
    zs = [z[i * Bh:(i + 1) * Bh] if z is not None else None for i in range(split)]
    forks = [torch.cuda.Stream() for _ in range(split - 1)]

    def step():
        cur = torch.cuda.current_stream()
        for s_ in forks:
            s_.wait_stream(cur)
        for i, h in enumerate(hs):
            st = cur if i == 0 else forks[i - 1]
            # the philox stream is keyed by (seed, element index): give each half its own key so halves do not repeat noise
            sd = 0 if pseed == 0 else (pseed + 2 * i) & 0xFFFFFFFFFFFFFFFF
            _lib.check(L.ddpm_sampler_step(h, xs[i].data_ptr(), zs[i].data_ptr() if zs[i] is not None else None, sd,
                                           C.c_void_p(st.cuda_stream)), "sampler_step")
        for s_ in forks:
            cur.wait_stream(s_)

    def draw():
        if z_out is not None:                   # block-size model: the reference draws in the outer shape
            z_out.normal_(generator=gen)
            _unshuffle_into(z, z_out, blk)
        elif z is not None:
            z.normal_(generator=gen)            # diffusion.py:155 - the reference's stream, drawn on the device

    def capture():
        graph = torch.cuda.CUDAGraph()
        if gen is not None and z is not None:
            graph.register_generator_state(gen)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                draw()
                step()
        torch.cuda.current_stream().wait_stream(side)
        return graph

    if ent is not None:
        # ONE graph launch per timestep: the captured step holds the noise draw (the generator is registered with the graph, so
        # every replay advances its Philox offset exactly like an eager normal_ call), the step-table fetch, the UNet forward and
        # the alpha/beta update fused into the final conv's gather.
        done = 0
        if ent["graph"] is None:
            draw(); step()                       # first use: one eager step (allocator warm-up), then capture (does not execute)
            done = 1
            ent["graph"] = capture()
        for _ in range(done, S):
            ent["graph"].replay()
        return x.clone()
    if use_graph and S > 1:                     # in-kernel Philox noise: the seed is a launch argument, so the graph is per call
        draw(); step()
        graph = capture()
        for _ in range(1, S):
            graph.replay()
    else:
        for _ in range(S):
            draw()
            step()
    return x
