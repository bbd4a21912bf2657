"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference,
tqch/ddpm-torch @ b60eb8d) on CPU fp32.  Run in the build container only:

    python oracle/gen_golden.py

The reference cannot travel to the GPU box, so its outputs are committed as small
fixtures; weights are NOT stored — they are regenerated from
``oracle.ddpm_ref.make_state_dict(cfg, seed)`` and loaded into the real reference
modules with ``load_state_dict(strict=True)`` (which also proves key/shape parity).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ddpm_ref as R  # noqa: E402


def import_reference():
    """The unmodified reference, imported through oracle/ref_loader.py (matplotlib stub, SURVEY.md §8(c))."""
    from oracle import ref_loader
    ref_loader.stage()
    return ref_loader.load()


def build_ref_unet(ddpm_torch, cfg, seed):
    c = R.normalize_cfg(cfg)
    m = ddpm_torch.UNet(in_channels=c["in_channels"], hid_channels=c["hid_channels"],
                        out_channels=c["out_channels"], ch_multipliers=c["ch_multipliers"],
                        num_res_blocks=c["num_res_blocks"], apply_attn=c["apply_attn"],
                        drop_rate=c["drop_rate"])
    sd = R.make_state_dict(cfg, seed)
    assert list(m.state_dict().keys()) == list(sd.keys()), "state_dict key order mismatch"
    m.load_state_dict(sd, strict=True)
    return m.eval(), sd


def inputs(cfg, B, H, W, seed, T=1000):
    g = torch.Generator().manual_seed(seed)
    x0 = torch.randn(B, cfg["in_channels"], H, W, generator=g)
    t = torch.randint(T, (B,), generator=g)
    noise = torch.randn(B, cfg["in_channels"], H, W, generator=g)
    return x0, t, noise


def sample_idx(n, k=64, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(n, (min(k, n),), generator=g)


def main():
    ddpm_torch, ddim = import_reference()
    out_dir = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out_dir, exist_ok=True)
    torch.manual_seed(0)
    torch.set_num_threads(os.cpu_count())

    betas = ddpm_torch.get_beta_schedule("linear", 1e-4, 0.02, 1000)

    # ---------------- schedule / coefficient tables (fp64, bit-exact) -----------------
    tabs = {}
    for vt in ("fixed-large", "fixed-small"):
        d = ddpm_torch.GaussianDiffusion(betas, "eps", vt, "mse")
        tabs[vt] = {k: getattr(d, k).clone() for k in (
            "betas", "alphas_bar", "sqrt_alphas_bar", "sqrt_one_minus_alphas_bar",
            "sqrt_recip_alphas_bar", "sqrt_recip_m1_alphas_bar", "posterior_var",
            "posterior_logvar_clipped", "posterior_mean_coef1", "posterior_mean_coef2",
            "fixed_model_var", "fixed_model_logvar")}
    for name, sched, S, eta in (("ddim_lin50_eta0", "linear", 50, 0.0), ("ddim_quad50_eta0", "quadratic", 50, 0.0),
                                ("ddim_lin100_eta0", "linear", 100, 0.0), ("ddim_lin10_eta1", "linear", 10, 1.0),
                                ("ddim_lin20_eta05", "linear", 20, 0.5)):
        sub = ddim.get_selection_schedule(sched, S, 1000)
        base = ddpm_torch.GaussianDiffusion(betas, "eps", "fixed-small", "mse")
        d = ddim.DDIM.from_ddpm(base, eta=eta, subsequence=sub)
        tabs[name] = {k: getattr(d, k).clone() for k in (
            "subsequence", "betas", "alphas_bar", "sqrt_alphas_bar", "sqrt_one_minus_alphas_bar",
            "sqrt_recip_alphas_bar", "sqrt_recip_m1_alphas_bar", "posterior_var",
            "posterior_logvar_clipped", "posterior_mean_coef1", "posterior_mean_coef2",
            "fixed_model_var", "fixed_model_logvar")}
        tabs[name]["model_var_type"] = d.model_var_type
    tabs["beta_schedules"] = {s: ddpm_torch.get_beta_schedule(s, 1e-4, 0.02, 1000)
                              for s in ("quad", "linear", "warmup10", "warmup50", "const", "jsd")}
    from ddpm_torch.functions import get_timestep_embedding
    tabs["temb128"] = get_timestep_embedding(torch.tensor([0, 1, 500, 999]), 128)
    tabs["temb32"] = get_timestep_embedding(torch.tensor([0, 1, 500, 999]), 32)
    torch.save(tabs, os.path.join(out_dir, "tables.pt"))
    print("tables.pt done")

    # ---------------- UNet forward / train_losses / backward ---------------------------
    cases = [
        ("tiny", R.TINY_CFG, 2, 16, 16, 11),
        ("small64", R.SMALL64_CFG, 4, 32, 32, 12),
        ("cifar10_bs4", R.CIFAR10_CFG, 4, 32, 32, 1234),
    ]
    for name, cfg, B, H, W, seed in cases:
        m, sd = build_ref_unet(ddpm_torch, cfg, seed)
        x0, t, noise = inputs(cfg, B, H, W, seed)
        t[0] = 0; t[-1] = 999
        diff = ddpm_torch.GaussianDiffusion(betas, "eps", "fixed-large", "mse")
        x_t = diff.q_sample(x0, t, noise)
        for p in m.parameters():
            p.requires_grad_(True)
        eps = m(x_t, t)
        losses = diff.train_losses(m, x0, t, noise)
        losses.mean().backward()
        gnorm = {k: p.grad.norm().item() for k, p in m.named_parameters()}
        gsample = {k: p.grad.flatten()[sample_idx(p.numel(), 64, i)].clone()
                   for i, (k, p) in enumerate(m.named_parameters())}
        # per-module goldens (first res block with a 1x1 skip, first attention block)
        fx = dict(cfg=dict(cfg), B=B, H=H, W=W, seed=seed, x0=x0, t=t, noise=noise, x_t=x_t,
                  eps=eps.detach().clone(), losses=losses.detach().clone(),
                  grad_norm=gnorm, grad_sample=gsample)
        # sampler steps with injected noise (fixed-large ancestral and fixed-small)
        with torch.no_grad():
            for vt in ("fixed-large", "fixed-small"):
                d = ddpm_torch.GaussianDiffusion(betas, "eps", vt, "mse")
                for tv in (0, 1, 500, 999):
                    tt = torch.full((B,), tv, dtype=torch.int64)
                    g = torch.Generator().manual_seed(777 + tv)
                    # reproduce p_sample_step's normal_ draw (diffusion.py:155) from a known generator
                    z = torch.empty_like(x_t).normal_(generator=torch.Generator().manual_seed(777 + tv))
                    xs = d.p_sample_step(m, x_t, tt, generator=g)
                    fx[f"pstep_{vt}_{tv}"] = xs.clone()
                    fx[f"pstep_noise_{tv}"] = z
            # 5-step DDIM (eta 0) and 4-step DDIM eta=1, full loop with seed
            for nm, sched, S, eta in (("ddim5_lin", "linear", 5, 0.0), ("ddim5_quad", "quadratic", 5, 0.0),
                                      ("ddim4_eta1", "linear", 4, 1.0)):
                sub = ddim.get_selection_schedule(sched, S, 1000)
                d = ddim.DDIM.from_ddpm(ddpm_torch.GaussianDiffusion(betas, "eps", "fixed-small", "mse"),
                                        eta=eta, subsequence=sub)
                xs = d.p_sample(m, shape=(B, cfg["in_channels"], H, W), device=torch.device("cpu"),
                                noise=noise.clone(), seed=4321)
                fx[nm] = xs.clone()
        torch.save(fx, os.path.join(out_dir, f"unet_{name}.pt"))
        print(f"unet_{name}.pt done  |eps|max={eps.abs().max():.4f} loss={losses.mean():.5f}")

    # ---------------- per-module goldens (reference modules directly) ------------------
    from ddpm_torch.models.unet import ResidualBlock, AttentionBlock
    mods = {}
    g = torch.Generator().manual_seed(5)

    def rnd(*s):
        return torch.randn(*s, generator=g)

    def fill(mod, shapes, seed):
        sd = {k[len("blk."):]: v for k, v in R.fill_params(shapes, seed).items()}
        assert list(mod.state_dict().keys()) == list(sd.keys())
        mod.load_state_dict(sd, strict=True)

    for nm, (ci, co, hw, B) in {"res_128_256": (128, 256, 16, 2), "res_128_128": (128, 128, 16, 2),
                                 "res_384_128": (384, 128, 8, 2)}.items():
        rb = ResidualBlock(ci, co, embed_dim=512, drop_rate=0.0).eval()
        fill(rb, R.res_block_shapes(ci, co, 512), 31)
        x, te = rnd(B, ci, hw, hw), rnd(B, 512)
        with torch.no_grad():
            y = rb(x.clone(), te)
        mods[nm] = dict(cin=ci, cout=co, seed=31, x=x, temb=te, y=y)
    for nm, (c, hw, B) in {"attn_128_8": (128, 8, 2), "attn_64_4": (64, 4, 2)}.items():
        ab = AttentionBlock(c).eval()
        fill(ab, R.attn_block_shapes(c), 32)
        x = rnd(B, c, hw, hw)
        with torch.no_grad():
            y = ab(x)
        mods[nm] = dict(c=c, seed=32, x=x, y=y)
    torch.save(mods, os.path.join(out_dir, "modules.pt"))
    print("modules.pt done")

    # ---------------- CelebA-HQ config, bs=1, 256x256: forward only ---------------------
    if os.environ.get("GOLDEN_HQ", "1") == "1":
        m, sd = build_ref_unet(ddpm_torch, R.CELEBAHQ_CFG, 99)
        x0, t, noise = inputs(R.CELEBAHQ_CFG, 1, 256, 256, 99)
        t[0] = 437
        with torch.no_grad():
            eps = m(x0, t)
        torch.save(dict(cfg=dict(R.CELEBAHQ_CFG), B=1, H=256, W=256, seed=99, x=x0, t=t,
                        eps=eps.to(torch.float16)), os.path.join(out_dir, "unet_celebahq_bs1.pt"))
        print(f"unet_celebahq_bs1.pt done |eps|max={eps.abs().max():.4f}")
    gen_optim(out_dir)
    gen_checkpoint(out_dir)
    gen_bpd(out_dir)


def gen_optim(out_dir):
    """clip_grad_norm_ + torch.optim.Adam + LambdaLR warm-up + the reference EMA class (utils/train.py:159-165,280-316)
    on a small parameter set for 8 steps; grads are deterministic.  Stored: initial params, per-step grads, and
    params / shadow / total-norm after every step."""
    ddpm_torch, _ = import_reference()
    from ddpm_torch.utils.train import EMA
    from torch.optim import Adam, lr_scheduler
    g = torch.Generator().manual_seed(4242)
    shapes = [(64,), (32, 16), (8, 3, 3, 3), (128,)]

    class M(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(s, generator=g) * 0.1) for s in shapes])
    m = M()
    hyper = dict(lr=2e-4, beta1=0.9, beta2=0.999, warmup=4, grad_norm=1.0, ema_decay=0.9999)
    opt = Adam(m.parameters(), lr=hyper["lr"], betas=(hyper["beta1"], hyper["beta2"]))
    sch = lr_scheduler.LambdaLR(opt, lr_lambda=lambda t: min((t + 1) / hyper["warmup"], 1.0))
    ema = EMA(m, decay=hyper["ema_decay"])
    fx = dict(hyper=hyper, shapes=shapes, p0=[p.detach().clone() for p in m.ps], grads=[], params=[], shadow=[], norms=[], lrs=[])
    for k in range(8):
        scale = [0.02, 5.0, 0.3, 1.0, 40.0, 0.001, 2.0, 0.7][k]           # both clipped and unclipped steps
        gs = [torch.randn(s, generator=g) * scale for s in shapes]
        for p, gr in zip(m.ps, gs):
            p.grad = gr.clone()
        fx["lrs"].append(opt.param_groups[0]["lr"])
        tn = torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=hyper["grad_norm"])
        opt.step(); opt.zero_grad(set_to_none=True); sch.step(); ema.update()
        fx["grads"].append(gs); fx["norms"].append(float(tn))
        fx["params"].append([p.detach().clone() for p in m.ps])
        fx["shadow"].append([ema.shadow[k_].clone() for k_, _ in m.named_parameters()])
    fx["ema_num_updates"] = ema.num_updates
    torch.save(fx, os.path.join(out_dir, "optim.pt"))
    print("optim.pt written; norms", [round(n, 4) for n in fx["norms"]], "lrs", fx["lrs"])


def gen_bpd(out_dir):
    """Bits-per-dim path of the UNMODIFIED reference (diffusion.py:107-138,203-250) on a toy non-native denoiser: every
    (model_mean_type, model_var_type) combination, loss terms at t = 0 / mid / T-1, the kl training loss, the prior term."""
    ddpm_torch, _ = import_reference()
    T = 20
    betas = ddpm_torch.get_beta_schedule("linear", 1e-4, 0.02, T)
    g = torch.Generator().manual_seed(31)
    x0 = (torch.rand(4, 3, 8, 8, generator=g) * 2 - 1).mul(127.5).round().div(127.5)       # 8-bit data rescaled to [-1, 1]
    noise = torch.randn(4, 3, 8, 8, generator=g)
    t = torch.tensor([0, 1, 9, T - 1])
    fx = dict(T=T, x0=x0, noise=noise, t=t, cases={})
    for mt in ("eps", "x_0", "mean"):
        for vt in ("fixed-small", "fixed-large"):      # "learned" cannot be constructed upstream (KeyError, diffusion.py:70-73)
            fn = R.toy_denoiser(3, 1, seed=5)
            d = ddpm_torch.GaussianDiffusion(betas=betas, model_mean_type=mt, model_var_type=vt, loss_type="kl")
            x_t = d.q_sample(x0, t, noise=noise)
            term, pred = d._loss_term_bpd(fn, x_0=x0, x_t=x_t, t=t, clip_denoised=True, return_pred=True)
            mean, var, logvar = d.p_mean_var(fn, x_t, t, clip_denoised=False, return_pred=False)
            fx["cases"][(mt, vt)] = dict(x_t=x_t, term=term, pred_x_0=pred, kl_loss=d.train_losses(fn, x0, t, noise=noise),
                                         mean=mean, var=var.expand_as(mean).clone(), logvar=logvar.expand_as(mean).clone())
            # (d._prior_bpd / d.calc_all_bpd raise upstream: the TorchScript-ed normal_kl rejects the float arguments of
            #  diffusion.py:249 and calc_all_bpd unpacks the shape tuple into B, diffusion.py:253 - nothing to pin there)
    torch.save(fx, os.path.join(out_dir, "bpd_toy.pt"))
    print("bpd_toy.pt written;", {k: [round(float(v), 4) for v in c["term"]] for k, c in list(fx["cases"].items())[:2]})


MICRO_CFG = dict(in_channels=3, hid_channels=32, out_channels=3, ch_multipliers=(1,), num_res_blocks=1, apply_attn=(False,), drop_rate=0.0)


def gen_checkpoint(out_dir):
    """A checkpoint in the reference's wire format (utils/train.py:264-276: {"model", "optimizer", "ema", "scheduler",
    "epoch"}), written after 3 real optimisation steps of the UNMODIFIED reference UNet / EMA with torch Adam + LambdaLR,
    with DDP-style "module." key prefixes on the model and EMA entries (what `train.py --distributed` writes and
    generate.py:83-85 / utils/train.py:255-259 strip)."""
    ddpm_torch, _ = import_reference()
    from ddpm_torch.utils.train import EMA
    from torch.optim import Adam, lr_scheduler
    m, sd = build_ref_unet(ddpm_torch, MICRO_CFG, 77)
    m.train()
    opt = Adam(m.parameters(), lr=2e-4, betas=(0.9, 0.999))
    sch = lr_scheduler.LambdaLR(opt, lr_lambda=lambda t: min((t + 1) / 5, 1.0))
    ema = EMA(m, decay=0.9999)
    diff = ddpm_torch.GaussianDiffusion(betas=ddpm_torch.get_beta_schedule("linear", 1e-4, 0.02, 1000), model_mean_type="eps",
                                        model_var_type="fixed-large", loss_type="mse")
    g = torch.Generator().manual_seed(5)
    for _ in range(3):
        x0 = torch.randn(2, 3, 16, 16, generator=g); t = torch.randint(1000, (2,), generator=g); nz = torch.randn(2, 3, 16, 16, generator=g)
        diff.train_losses(m, x0, t, nz).mean().backward()
        torch.nn.utils.clip_grad_norm_(m.parameters(), max_norm=1.0)
        opt.step(); opt.zero_grad(set_to_none=True); sch.step(); ema.update()
    pre = lambda d: {"module." + k: v for k, v in d.items()}
    esd = ema.state_dict()
    chk = {"model": pre(m.state_dict()), "optimizer": opt.state_dict(),
           "ema": {"decay": esd["decay"], "shadow": pre(esd["shadow"]), "num_updates": esd["num_updates"]},
           "scheduler": sch.state_dict(), "epoch": 7}
    torch.save(dict(cfg=MICRO_CFG, seed=77, chkpt=chk), os.path.join(out_dir, "checkpoint_micro.pt"))
    print("checkpoint_micro.pt written; scheduler", {k: v for k, v in chk["scheduler"].items() if k != "lr_lambdas"})


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "bpd":
        gen_bpd(os.path.join(ROOT, "tests", "golden")); sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "checkpoint":
        gen_checkpoint(os.path.join(ROOT, "tests", "golden")); sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "optim":
        gen_optim(os.path.join(ROOT, "tests", "golden")); sys.exit(0)
    main()
