"""Block-size models on the engine (train.py:63-73: ModelWrapper(UNet(C*b*b, ..., C*b*b), PixelUnshuffle(b), PixelShuffle(b))):
wrapped forward, native training and sampling through the wrapper, against the golden of the unmodified reference, the oracle
(fp32, TF32 off) and the generic torch path.  Bars are DESIGN.md §2's; measured values are printed (run with -s)."""
import os
import socket

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import ddpm_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


def check_device_flag():
    from ddpm_torch_b200 import _lib
    assert _lib.lib().ddpm_device_error_flag() == 0


def build(cfg, seed, b, train=False, generic=False):
    """(engine UNet, wrapper, oracle state_dict on the device).  generic=True wraps with a transform the native dispatch does not
    recognise (same arithmetic), which forces the generic torch path over the same engine UNet."""
    import ddpm_torch_b200 as D
    c = R.normalize_cfg(cfg)
    m = D.UNet(c["in_channels"], c["hid_channels"], c["out_channels"], c["ch_multipliers"], c["num_res_blocks"], c["apply_attn"],
               drop_rate=0.0)
    sd = R.make_state_dict(cfg, seed)
    m.load_state_dict(sd)
    m = m.to(DEV).train(train)
    pre = nn.Sequential(nn.PixelUnshuffle(b)) if generic else nn.PixelUnshuffle(b)
    return m, D.ModelWrapper(m, pre, nn.PixelShuffle(b)), {k: v.to(DEV) for k, v in sd.items()}


def oracle_eps(sd, cfg, b, x, t):
    return F.pixel_shuffle(R.unet_forward(sd, cfg, F.pixel_unshuffle(x, b), t), b)


def wide(cfg, ch):
    return dict(cfg, in_channels=ch, out_channels=ch)


def betas(T=1000):
    import ddpm_torch_b200 as D
    return D.get_beta_schedule("linear", 1e-4, 0.02, T)


# (name, cfg, block size, images, outer H = W)
FWD_CASES = [("cifar_b2_bs128", wide(R.CIFAR10_CFG, 12), 2, 128, 32),
             ("celebahq_b2_bs2", wide(R.CELEBAHQ_CFG, 12), 2, 2, 256),
             ("small64_1ch_b4", wide(R.SMALL64_CFG, 16), 4, 1, 64)]


def test_wrapped_forward_vs_golden_and_oracle(golden):
    fx = golden("unet_block2_small64.pt")
    m, w, sd = build(fx["cfg"], fx["seed"], fx["block_size"])
    x, t = fx["x_t"].to(DEV), fx["t"].to(DEV)
    with torch.no_grad():
        eps = w(x, t)
        ref = oracle_eps(sd, fx["cfg"], fx["block_size"], x, t)
    check_device_flag()
    r1, r2 = rel(eps, ref), rel(eps.cpu(), fx["eps"])
    print(f"\n[block2 small64] eps rel-L2 vs oracle {r1:.3e}, vs reference golden {r2:.3e}")
    assert eps.shape == x.shape and r1 <= 1e-2 and r2 <= 1e-2


@pytest.mark.parametrize("name,cfg,b,B,HW", FWD_CASES)
def test_wrapped_forward_vs_oracle(name, cfg, b, B, HW):
    m, w, sd = build(cfg, 17, b)
    g = torch.Generator(DEV).manual_seed(5)
    x = torch.randn(B, cfg["in_channels"] // (b * b), HW, HW, device=DEV, generator=g)
    t = torch.randint(1000, (B,), device=DEV, generator=g)
    with torch.no_grad():
        eps = w(x, t)
        ref = oracle_eps(sd, cfg, b, x, t)
    check_device_flag()
    r = rel(eps, ref)
    print(f"\n[{name}] eps rel-L2 vs oracle {r:.3e}")
    assert eps.shape == x.shape and r <= 1e-2


def grad_report(tag, m, sdg, losses, lref):
    lr = ((losses - lref).abs().max() / lref.abs().max()).item()
    gm = torch.cat([p.grad.flatten() for p in m.parameters()])
    gr = torch.cat([sdg[k].grad.flatten() for k, _ in m.named_parameters()])
    worst, bad = 1.0, []
    for k, p in m.named_parameters():
        a, b_ = p.grad.flatten().double(), sdg[k].grad.flatten().double()
        if b_.norm() < 1e-6 * gr.norm():
            continue
        cos = (a @ b_ / (a.norm() * b_.norm()).clamp_min(1e-30)).item()
        worst = min(worst, cos)
        if cos < 0.995:
            bad.append((k, cos))
    print(f"[{tag}] loss rel {lr:.3e}; flat grad rel-L2 {rel(gm, gr):.3e}; worst per-tensor cosine {worst:.5f}")
    assert lr <= 1e-2 and rel(gm, gr) <= 5e-2 and not bad, bad[:5]


@pytest.mark.parametrize("generic", [False, True])
def test_train_losses_through_the_wrapper(golden, generic):
    import ddpm_torch_b200 as D
    fx = golden("unet_block2_small64.pt")
    cfg, b = fx["cfg"], fx["block_size"]
    m, w, sd = build(cfg, fx["seed"], b, train=True, generic=generic)
    assert (D.GaussianDiffusion(betas(), "eps", "fixed-large", "mse")._fast_ok(w)[0] is None) == generic
    diff = D.GaussianDiffusion(betas(), "eps", "fixed-large", "mse")
    x0, t, noise = fx["x0"].to(DEV), fx["t"].to(DEV), fx["noise"].to(DEV)
    losses = diff.train_losses(w, x0, t, noise)
    assert losses.shape == (x0.shape[0],)
    losses.mean().backward()
    check_device_flag()
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    rd = R.RefDiffusion(R.get_beta_schedule("linear", 1e-4, 0.02, 1000), "fixed-large")
    lref = rd.train_losses(lambda x, tt: oracle_eps(sdg, cfg, b, x, tt), x0, t, noise)
    lref.mean().backward()
    tag = "generic" if generic else "native"
    print(f"\n[block2 {tag}] loss vs reference golden: max rel {((losses.cpu() - fx['losses']).abs() / fx['losses'].abs()).max().item():.3e}")
    grad_report(f"block2 {tag} vs oracle", m, sdg, losses, lref)
    assert ((losses.detach().cpu() - fx["losses"]).abs() / fx["losses"].abs()).max().item() <= 1e-2
    for k, p in m.named_parameters():
        gn = fx["grad_norm"][k]
        if gn > 1e-3:
            assert abs(p.grad.norm().item() - gn) / gn < 0.1, k


def test_sixteen_channel_train_losses_vs_oracle():
    import ddpm_torch_b200 as D
    cfg = wide(R.SMALL64_CFG, 16)
    m, w, sd = build(cfg, 23, 4, train=True)
    g = torch.Generator(DEV).manual_seed(9)
    x0 = torch.randn(2, 1, 64, 64, device=DEV, generator=g); t = torch.randint(1000, (2,), device=DEV, generator=g)
    noise = torch.randn(2, 1, 64, 64, device=DEV, generator=g)
    losses = D.GaussianDiffusion(betas(), "eps", "fixed-large", "mse").train_losses(w, x0, t, noise)
    losses.mean().backward()
    check_device_flag()
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    lref = R.RefDiffusion(R.get_beta_schedule("linear", 1e-4, 0.02, 1000), "fixed-large").train_losses(
        lambda x, tt: oracle_eps(sdg, cfg, 4, x, tt), x0, t, noise)
    lref.mean().backward()
    grad_report("16ch b4", m, sdg, losses, lref)


def test_teacher_forced_sampler_steps_vs_golden(golden):
    """One reverse step from the golden x_t with the golden's injected noise, through the wrapped engine model."""
    import ddpm_torch_b200 as D
    fx = golden("unet_block2_small64.pt")
    m, w, _ = build(fx["cfg"], fx["seed"], fx["block_size"])
    x_t, B = fx["x_t"].to(DEV), fx["B"]
    worst = 0.0
    for vt in ("fixed-large", "fixed-small"):
        d = D.GaussianDiffusion(betas(), "eps", vt, "mse")
        for tv in (0, 1, 500, 999):
            tt = torch.full((B,), tv, dtype=torch.int64, device=DEV)
            with torch.no_grad():
                mean, _, logvar = d.p_mean_var(w, x_t, tt, True, False)
            nz = (tt > 0).reshape(-1, 1, 1, 1).float()
            xs = mean + nz * torch.exp(0.5 * logvar) * fx[f"pstep_noise_{tv}"].to(DEV)
            ref = fx[f"pstep_{vt}_{tv}"]
            err, scale = (xs.cpu() - ref).abs().max().item(), ref.abs().max().item()
            worst = max(worst, err / max(scale, 1.0))
            assert err < 5e-2 * max(scale, 1.0), (vt, tv, err, scale)
    print(f"\n[block2 teacher-forced steps] worst Linf / scale {worst:.3e}")
    check_device_flag()


def test_ddim5_vs_golden(golden):
    import ddpm_torch_b200 as D
    fx = golden("unet_block2_small64.pt")
    m, w, _ = build(fx["cfg"], fx["seed"], fx["block_size"])
    sub = D.get_selection_schedule("linear", 5, 1000)
    dd = D.DDIM.from_ddpm(D.GaussianDiffusion(betas(), "eps", "fixed-small", "mse"), eta=0.0, subsequence=sub)
    for use_graph in (False, True):
        xs = dd.p_sample(w, shape=tuple(fx["noise"].shape), device=torch.device(DEV), noise=fx["noise"].to(DEV), seed=4321,
                         use_graph=use_graph)
        assert xs.shape == fx["noise"].shape
        dlt = (xs.cpu() - fx["ddim5_lin"]).abs()
        l1, frac = dlt.mean().item(), (dlt > 0.1).float().mean().item()
        print(f"\n[block2 ddim5] graph={use_graph} vs reference golden: pixel L1 {l1:.3e}, frac(|d|>0.1) {frac:.4f}")
        assert l1 <= 2e-2 and frac <= 0.03
    check_device_flag()


def test_native_chain_matches_generic_chain():
    """T = 20 ancestral chain with the same seed: the native loop draws every step's noise in the outer shape from the caller's
    generator, exactly as the generic loop (the reference) does."""
    import ddpm_torch_b200 as D
    cfg = wide(R.SMALL64_CFG, 12)
    m, w, _ = build(cfg, 31, 2)
    _, wg, _ = build(cfg, 31, 2, generic=True)
    d = D.GaussianDiffusion(betas(20), "eps", "fixed-large", "mse")
    shape = (8, 3, 32, 32)
    ref = d.p_sample(wg, shape=shape, device=torch.device(DEV), seed=11)
    for use_graph in (False, True):
        xs = d.p_sample(w, shape=shape, device=torch.device(DEV), seed=11, use_graph=use_graph)
        err = (xs - ref).abs().max().item()
        print(f"\n[block2 T=20 chain] native graph={use_graph} vs generic: pixel Linf {err:.3e}")
        assert xs.shape == shape and err <= 5e-2
    xa, pa = d.p_sample_progressive(w, shape, device=torch.device(DEV), seed=11, pred_freq=5)
    xb, pb = d.p_sample_progressive(wg, shape, device=torch.device(DEV), seed=11, pred_freq=5)
    assert xa.shape == shape and pa.shape == (4,) + shape
    e1, e2 = (xa - xb).abs().max().item(), (pa - pb).abs().max().item()
    print(f"[block2 progressive] native vs generic: sample Linf {e1:.3e}, predictions Linf {e2:.3e}")
    assert e1 <= 5e-2 and e2 <= 5e-2
    check_device_flag()


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _ddp_worker(rank, world, port, ret):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    import ddpm_torch_b200 as D
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    cfg = wide(R.SMALL64_CFG, 12)
    c = R.normalize_cfg(cfg)
    inner = D.UNet(12, c["hid_channels"], 12, c["ch_multipliers"], c["num_res_blocks"], c["apply_attn"], drop_rate=0.0)
    inner.load_state_dict(R.make_state_dict(cfg, 12))
    inner = inner.to(dev).train()
    wrapped = D.ModelWrapper(inner, nn.PixelUnshuffle(2), nn.PixelShuffle(2))
    model = DDP(wrapped, device_ids=[0])                          # train.py:110
    diff = D.GaussianDiffusion(betas(), "eps", "fixed-large", "mse")
    g = torch.Generator(dev).manual_seed(100 + rank)              # different data per rank
    x0 = torch.randn(4, 3, 32, 32, device=dev, generator=g); t = torch.randint(1000, (4,), device=dev, generator=g)
    nz = torch.randn(4, 3, 32, 32, device=dev, generator=g)
    inner.zero_grad()
    diff.train_losses(wrapped, x0, t, nz).mean().backward()       # local gradient: the wrapper alone does not reduce
    local = torch.cat([p.grad.flatten() for p in inner.parameters()]).clone()
    inner.zero_grad()
    diff.train_losses(model, x0, t, nz).mean().backward()
    red = torch.cat([p.grad.flatten() for p in inner.parameters()]).clone()
    locs = [torch.empty_like(local) for _ in range(world)]; reds = [torch.empty_like(red) for _ in range(world)]
    dist.all_gather(locs, local); dist.all_gather(reds, red)
    mean = sum(locs) / world
    r = lambda a, b: ((a.double() - b.double()).norm() / b.double().norm()).item()
    ret[rank] = dict(equal=bool(torch.equal(reds[0], reds[1])), vs_mean=r(red, mean), vs_local=r(red, local), local_diff=r(locs[0], locs[1]))
    dist.barrier()
    dist.destroy_process_group()


def test_ddp_wrapped_block_model_averages_gradients():
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    procs = [ctx.Process(target=_ddp_worker, args=(r, world, port, ret)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(600)
        assert p.exitcode == 0
    for r in range(world):
        d = ret[r]
        print(f"\n[block2 ddp rank {r}] {d}")
        assert d["equal"], "replicas hold different gradients"
        assert d["vs_mean"] < 2e-2
        assert d["local_diff"] > 0.1 and d["vs_local"] > 0.05
