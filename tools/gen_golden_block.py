"""Generate tests/golden/unet_block2_small64.pt: a block-size model of the UNMODIFIED reference on CPU fp32.

    python tools/gen_golden_block.py

The model is what train.py:63-73 builds for RGB at block size 2: the reference UNet with in_channels = out_channels = 12 inside
the reference ModelWrapper(model, PixelUnshuffle(2), PixelShuffle(2)) (utils/train.py:349-367), on a SMALL64-like config
(64 hidden channels: tensor-core geometry) at 3x32x32 outside / 12x16x16 inside, 4 images, with the t[0] = 0, t[-1] = 999
convention of oracle/gen_golden.py's unet_*.pt.  Weights are NOT stored: they are oracle.ddpm_ref.make_state_dict(BLOCK_CFG,
SEED).  Stored: the wrapped eps, per-sample train_losses, per-parameter gradient norms and samples, teacher-forced
p_sample_step outputs with injected noise at t in {0, 1, 500, 999} for both fixed variances, and a seeded 5-step DDIM loop.
Existing goldens are not touched.
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ddpm_ref as R  # noqa: E402
from oracle.gen_golden import build_ref_unet, import_reference, sample_idx  # noqa: E402

BLOCK = 2
BLOCK_CFG = dict(R.SMALL64_CFG, in_channels=3 * BLOCK * BLOCK, out_channels=3 * BLOCK * BLOCK)
SEED, B, H, W = 21, 4, 32, 32


def ref_wrapper(ddpm_torch, model, b):
    """The reference's ModelWrapper; the same three calls in the same order if its module cannot be imported."""
    try:
        from ddpm_torch.utils.train import ModelWrapper
        return ModelWrapper(model, torch.nn.PixelUnshuffle(b), torch.nn.PixelShuffle(b))
    except ImportError:
        pre, post = torch.nn.PixelUnshuffle(b), torch.nn.PixelShuffle(b)
        return lambda x, *a, **k: post(model(pre(x), *a, **k))


def gen_block(out_dir):
    ddpm_torch, ddim = import_reference()
    torch.manual_seed(0)
    betas = ddpm_torch.get_beta_schedule("linear", 1e-4, 0.02, 1000)
    m, _ = build_ref_unet(ddpm_torch, BLOCK_CFG, SEED)
    w = ref_wrapper(ddpm_torch, m, BLOCK)
    g = torch.Generator().manual_seed(SEED)
    x0 = torch.randn(B, 3, H, W, generator=g)
    t = torch.randint(1000, (B,), generator=g)
    noise = torch.randn(B, 3, H, W, generator=g)
    t[0] = 0; t[-1] = 999
    diff = ddpm_torch.GaussianDiffusion(betas, "eps", "fixed-large", "mse")
    x_t = diff.q_sample(x0, t, noise)
    for p in m.parameters():
        p.requires_grad_(True)
    eps = w(x_t, t)
    losses = diff.train_losses(w, x0, t, noise)
    losses.mean().backward()
    fx = dict(cfg=dict(BLOCK_CFG), block_size=BLOCK, B=B, H=H, W=W, seed=SEED, x0=x0, t=t, noise=noise, x_t=x_t,
              eps=eps.detach().clone(), losses=losses.detach().clone(),
              grad_norm={k: p.grad.norm().item() for k, p in m.named_parameters()},
              grad_sample={k: p.grad.flatten()[sample_idx(p.numel(), 64, i)].clone() for i, (k, p) in enumerate(m.named_parameters())})
    with torch.no_grad():
        for vt in ("fixed-large", "fixed-small"):
            d = ddpm_torch.GaussianDiffusion(betas, "eps", vt, "mse")
            for tv in (0, 1, 500, 999):
                tt = torch.full((B,), tv, dtype=torch.int64)
                # p_sample_step draws its noise with normal_ in the outer shape (diffusion.py:155): record that draw
                fx[f"pstep_noise_{tv}"] = torch.empty_like(x_t).normal_(generator=torch.Generator().manual_seed(777 + tv))
                fx[f"pstep_{vt}_{tv}"] = d.p_sample_step(w, x_t, tt, generator=torch.Generator().manual_seed(777 + tv)).clone()
        sub = ddim.get_selection_schedule("linear", 5, 1000)
        d = ddim.DDIM.from_ddpm(ddpm_torch.GaussianDiffusion(betas, "eps", "fixed-small", "mse"), eta=0.0, subsequence=sub)
        fx["ddim5_lin"] = d.p_sample(w, shape=(B, 3, H, W), device=torch.device("cpu"), noise=noise.clone(), seed=4321).clone()
    path = os.path.join(out_dir, "unet_block2_small64.pt")
    torch.save(fx, path)
    print(f"{path} written ({os.path.getsize(path)} bytes) |eps|max={eps.abs().max():.4f} loss={losses.mean():.5f}")


if __name__ == "__main__":
    gen_block(os.path.join(ROOT, "tests", "golden"))
