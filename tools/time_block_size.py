"""Cost of block-size models (train.py --block-size b: UNet(C*b*b, ...) on pixel_unshuffle(x, b) at 1/b the resolution) against
b = 1, through the public API (ModelWrapper + GaussianDiffusion / DDIM, pixel (un)shuffle copies included):

* CelebA-HQ 256^2 (configs/celebahq.json): training step at 4 images (train_losses + backward), DDIM-100 (eta 0) at 8 images;
* CIFAR-10 32^2 (configs/cifar10.json, dropout 0.1): training step at 128 images.

Same conventions as bench.py's hq_train / hq_ddim100: uniform fan-in weights, seeded inputs, warm-up, CUDA events around the
timed window.  The GPU name and power limit are read in the same run and written beside the numbers.

    python tools/time_block_size.py --out profiles/r03_block_size.json
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402

import ddpm_torch_b200 as D  # noqa: E402
from ddpm_torch_b200 import _lib  # noqa: E402
from oracle import ddpm_ref as R  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0)}


def make(cfg, b, dev):
    c = R.normalize_cfg(cfg)
    ch = c["in_channels"] * b * b
    m = D.UNet(ch, c["hid_channels"], ch, c["ch_multipliers"], c["num_res_blocks"], c["apply_attn"], drop_rate=c["drop_rate"])
    m = m.to(dev).train()
    with torch.no_grad():
        gi = torch.Generator(device=dev).manual_seed(7)
        for p in m.parameters():
            if p.ndim >= 2:
                p.copy_((torch.rand(p.shape, device=dev, generator=gi) * 2 - 1) * (3.0 / p[0].numel()) ** 0.5)
    return m, (m if b == 1 else D.ModelWrapper(m, nn.PixelUnshuffle(b), nn.PixelShuffle(b)))


def time_train(cfg, b, B, HW, dev, steps, warmup):
    m, w = make(cfg, b, dev)
    diff = D.GaussianDiffusion(D.get_beta_schedule("linear", 1e-4, 0.02, 1000), "eps", "fixed-small", "mse")
    g = torch.Generator(device=dev).manual_seed(200)
    x0 = torch.rand(B, 3, HW, HW, device=dev, generator=g) * 2 - 1
    t = torch.randint(1000, (B,), device=dev, generator=g); nz = torch.randn(B, 3, HW, HW, device=dev, generator=g)

    def step():
        m.zero_grad()
        diff.train_losses(w, x0, t, nz).mean().backward()
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    assert all(torch.isfinite(p.grad).all() for p in m.parameters())
    return {"block_size": b, "images": B, "unet_input": [B, 3 * b * b, HW // b, HW // b], "ms_per_step": ms,
            "images_per_s": B / ms * 1e3, "steps": steps, "warmup": warmup}


def time_ddim(cfg, b, B, HW, dev, S=100):
    m, w = make(cfg, b, dev)
    m.eval()
    ddim = D.DDIM.from_ddpm(D.GaussianDiffusion(D.get_beta_schedule("linear", 1e-4, 0.02, 1000), "eps", "fixed-small", "mse"),
                            eta=0.0, subsequence=D.get_selection_schedule("linear", S, 1000))
    ddim.p_sample(w, shape=(B, 3, HW, HW), device=dev, seed=3)            # warm-up (plan, step graph)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    x = ddim.p_sample(w, shape=(B, 3, HW, HW), device=dev, seed=5)
    e1.record(); torch.cuda.synchronize()
    s = e0.elapsed_time(e1) * 1e-3
    assert torch.isfinite(x).all()
    return {"block_size": b, "images": B, "unet_input": [B, 3 * b * b, HW // b, HW // b], "steps": S, "seconds_per_batch": s,
            "ms_per_step": s * 1e3 / S, "images_per_s": B / s}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r03_block_size.json")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(), "api": "public: ModelWrapper + GaussianDiffusion.train_losses / DDIM.p_sample, pixel (un)shuffle included"}
    for b in (1, 2):
        res[f"celebahq256_train_bs4_b{b}"] = time_train(R.CELEBAHQ_CFG, b, 4, 256, dev, a.steps, a.warmup)
        print(res[f"celebahq256_train_bs4_b{b}"], flush=True)
        torch.cuda.empty_cache()
        res[f"celebahq256_ddim100_bs8_b{b}"] = time_ddim(R.CELEBAHQ_CFG, b, 8, 256, dev)
        print(res[f"celebahq256_ddim100_bs8_b{b}"], flush=True)
        torch.cuda.empty_cache()
    for b in (1, 2):
        res[f"cifar32_train_bs128_b{b}"] = time_train(R.CIFAR10_CFG, b, 128, 32, dev, a.steps, a.warmup)
        print(res[f"cifar32_train_bs128_b{b}"], flush=True)
        torch.cuda.empty_cache()
    assert _lib.lib().ddpm_device_error_flag() == 0
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("written", a.out)


if __name__ == "__main__":
    main()
