"""Block-size models (train.py:63-73: UNet(C*b*b, ..., C*b*b) inside ModelWrapper(PixelUnshuffle(b), PixelShuffle(b))) without a
GPU: the oracle composed with the pixel (un)shuffles reproduces the reference golden, the engine plans 5..16 image channels on
the tensor-core narrow convolutions and refuses what it cannot run, plans with <= 4 channels keep their launch lists, and the
mirror's wrapper has the reference's state_dict keys."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from oracle import ddpm_ref as R


@pytest.fixture(scope="module")
def L():
    from ddpm_torch_b200 import _lib
    return _lib.lib()


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def _handle(L, cfg, cin, cout, hid=None):
    from ddpm_torch_b200 import _lib
    c = R.normalize_cfg(cfg)
    u = _lib.UnetCfg()
    u.in_channels, u.hid_channels, u.out_channels = cin, hid or c["hid_channels"], cout
    u.levels, u.num_res_blocks, u.temb_dim, u.drop_rate = len(c["ch_multipliers"]), c["num_res_blocks"], 0, c["drop_rate"]
    for i, m in enumerate(c["ch_multipliers"]):
        u.ch_mult[i] = m; u.attn[i] = int(c["apply_attn"][i])
    h = C.c_void_p()
    assert L.ddpm_unet_create(C.byref(u), C.byref(h)) == 0, L.ddpm_last_error()
    return h


def _plan(L, h, B, H, W, train):
    ws = L.ddpm_unet_workspace_bytes(h, B, H, W, int(train))
    nf, nb, npk = C.c_int(), C.c_int(), C.c_int()
    L.ddpm_unet_launch_counts(h, C.byref(nf), C.byref(nb), C.byref(npk))
    return ws, (nf.value, nb.value, npk.value)


def test_oracle_with_pixel_shuffle_matches_reference_golden(golden):
    fx = golden("unet_block2_small64.pt")
    b, cfg = fx["block_size"], fx["cfg"]
    sd = R.make_state_dict(cfg, fx["seed"])
    with torch.no_grad():
        eps = F.pixel_shuffle(R.unet_forward(sd, cfg, F.pixel_unshuffle(fx["x_t"], b), fx["t"]), b)
    r = rel(eps, fx["eps"])
    print(f"\n[block2 small64] oracle o pixel (un)shuffle vs reference golden: eps rel-L2 {r:.3e}")
    assert eps.shape == fx["x_t"].shape and r < 1e-5


@pytest.mark.parametrize("cfg,B,HW", [(R.CIFAR10_CFG, 128, 16), (R.CELEBAHQ_CFG, 4, 128)])
@pytest.mark.parametrize("ch", [12, 16])
def test_wide_image_channels_plan_on_the_tensor_cores(L, cfg, B, HW, ch):
    wcfg = dict(cfg, in_channels=ch, out_channels=ch)
    h = _handle(L, cfg, ch, ch)
    need = L.ddpm_unet_workspace_bytes(h, B, HW, HW, 1)
    assert need > 0, L.ddpm_last_error()
    nf, nb, ntc, ng = C.c_int(), C.c_int(), C.c_int(), C.c_int(); ff, bf = C.c_double(), C.c_double()
    L.ddpm_unet_plan_stats(h, C.byref(nf), C.byref(nb), C.byref(ntc), C.byref(ng), C.byref(ff), C.byref(bf))
    ref = R.fwd_flops_per_image(wcfg, HW, HW)
    assert abs(ff.value / B - ref) / ref < 1e-6
    assert 1.9 < bf.value / ff.value < 2.2
    assert ntc.value > 5 * ng.value
    L.ddpm_unet_destroy(h)


def test_unsupported_image_channels_are_errors_not_aborts(L):
    h = _handle(L, R.CIFAR10_CFG, 17, 17)
    assert L.ddpm_unet_workspace_bytes(h, 4, 32, 32, 1) < 0
    assert b"1..16" in L.ddpm_last_error()
    L.ddpm_unet_destroy(h)
    h = _handle(L, R.CIFAR10_CFG, 12, 12, hid=96)       # 5..16 channels exist only on the tensor-core routes (hid % 64 == 0)
    assert L.ddpm_unet_workspace_bytes(h, 4, 32, 32, 1) < 0
    assert b"tensor-core" in L.ddpm_last_error() and b"hid_channels" in L.ddpm_last_error()
    L.ddpm_unet_destroy(h)
    h = _handle(L, R.CIFAR10_CFG, 3, 12)
    assert L.ddpm_unet_workspace_bytes(h, 4, 32, 32, 0) > 0           # either side may be wide on its own
    L.ddpm_unet_destroy(h)


@pytest.mark.parametrize("cin,cout,B,train,counts", [
    (3, 3, 256, False, (137, 0, 4)),        # bench.py sampler shape
    (3, 3, 128, True, (146, 378, 5)),       # bench.py training shape
    (4, 4, 128, True, (145, 376, 3)),       # 4 channels: CUDA-core out_conv
])
def test_narrow_plans_keep_their_launch_lists(L, cin, cout, B, train, counts):
    h = _handle(L, R.CIFAR10_CFG, cin, cout)
    ws, got = _plan(L, h, B, 32, 32, train)
    assert ws > 0 and got == counts
    L.ddpm_unet_destroy(h)


def test_wrapper_state_dict_keys_are_the_references():
    import ddpm_torch_b200 as D
    from oracle import ref_loader
    if not ref_loader.available():
        pytest.skip("reference not staged (build() stages it)")
    ddpm_torch, _ = ref_loader.load()
    from ddpm_torch.utils.train import ModelWrapper
    cfg = dict(R.SMALL64_CFG, in_channels=12, out_channels=12)
    c = R.normalize_cfg(cfg)
    args = (12, c["hid_channels"], 12, c["ch_multipliers"], c["num_res_blocks"], c["apply_attn"])
    mine = D.ModelWrapper(D.UNet(*args), torch.nn.PixelUnshuffle(2), torch.nn.PixelShuffle(2))
    ref = ModelWrapper(ddpm_torch.UNet(*args), torch.nn.PixelUnshuffle(2), torch.nn.PixelShuffle(2))
    keys = list(ref.state_dict().keys())
    assert keys[0].startswith("_model.") and list(mine.state_dict().keys()) == keys
    mine.load_state_dict(ref.state_dict())                       # a block-size checkpoint loads as is
    assert all(torch.equal(v, ref.state_dict()[k]) for k, v in mine.state_dict().items())


def test_native_dispatch_recognises_only_pixel_shuffle_wrappers():
    import torch.nn as nn
    import ddpm_torch_b200 as D
    from ddpm_torch_b200.diffusion import _native
    u = D.UNet(12, 64, 12, (1, 2), 1, (False, True))
    assert _native(D.ModelWrapper(u, nn.PixelUnshuffle(2), nn.PixelShuffle(2))) == (u, 2)

    class Holder(nn.Module):                   # DDP-like `.module` holder around the wrapper (train.py:110)
        def __init__(self, m):
            super().__init__()
            self.module = m
    assert _native(Holder(D.ModelWrapper(u, nn.PixelUnshuffle(2), nn.PixelShuffle(2)))) == (u, 2)
    assert _native(u) == (u, 1)
    for w in (D.ModelWrapper(u, nn.Sequential(nn.PixelUnshuffle(2)), nn.PixelShuffle(2)),
              D.ModelWrapper(u, nn.PixelUnshuffle(2), nn.PixelShuffle(4)),
              D.ModelWrapper(u), D.ModelWrapper(nn.Identity(), nn.PixelUnshuffle(2), nn.PixelShuffle(2))):
        assert _native(w) == (None, 1)
