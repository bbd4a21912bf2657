#!/usr/bin/env python
"""bench.py — headline metric of BASELINE.json: UNet fwd+bwd images/sec (CIFAR-10 config, bs=128 per GPU, training
mode, synthetic 3x32x32) on N B200s, plus p_sample-loop images/sec (bs=256) at N=1.

    python bench.py [--gpus N --steps K --warmup W]           # this framework (sm_100a engine through the C ABI)
    python bench.py --impl reference [...]                     # the UNMODIFIED reference (oracle/_ref) on the host CPU
    python bench.py [...] --dump-outputs DIR                   # + the last timed step's losses / gradients as DIR/*.npy

One JSON line on stdout (rank 0).  `value` = whole-job images/s with inputs resident in HBM; `e2e` = the same step
driven through the public Python API with the batch coming from pinned host memory and the loss read back.
A "step" = weight re-pack + q_sample + UNet forward + MSE + full backward (grads of all 304 tensors)
(+ the NCCL all-reduce (mean) of the flat gradient buffer when N > 1, issued chunk by chunk on a communication stream as the
backward pass completes each level group).  Optimiser/EMA are outside the metric.
Extra keys at every N (BASELINE configs 3-5): `sampler` (CIFAR bs=256 per GPU, DDIM-50 + ancestral-1000), `hq_train`
(celebahq.json 3x256x256, 4 images per GPU, incl. the 455 MB all-reduce), `hq_ddim100` (8 images per GPU, no collective);
at N=1 also `vs_stock_cuda` (the unmodified reference's torch-CUDA step on the same B200 - north_star's >=10x denominator).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CIFAR = dict(in_channels=3, hid_channels=128, out_channels=3, ch_multipliers=(1, 2, 2, 2), num_res_blocks=2,
             apply_attn=(False, True, False, False), drop_rate=0.1)
HQ = dict(in_channels=3, hid_channels=128, out_channels=3, ch_multipliers=(1, 1, 2, 2, 4, 4), num_res_blocks=2,
          apply_attn=(False, False, False, False, True, False), drop_rate=0.0)          # configs/celebahq.json
FWD_GFLOP_PER_IMG = 12.444          # SURVEY.md section 8(d): 2*MAC of convs + linears + attention matmuls
TRAIN_GFLOP_PER_IMG = 3 * FWD_GFLOP_PER_IMG
HQ_FWD_GFLOP_PER_IMG = 497.03
# torch CPU threads for the reference arm: measured on the 128-core GPU-box host (tools/cpu_threads.py, bs=32 fwd+bwd):
# 8 -> 25, 16 -> 43.5, 32 -> 35, 64 -> 18, 128 -> 0.1 images/s; 16 is the fastest, so "all the threads it can use" = 16.
CPU_THREADS = min(16, os.cpu_count() or 1)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(burst=d["bf16_tflops"], sustained=d["bf16_tflops_sustained"], hbm=d["hbm_gbs"], src="measured")
    return dict(burst=1590.0, sustained=1400.0, hbm=6650.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.stop_flag, self.index = [], False, index
        self.nv = None
        try:                                   # NVML is initialised HERE, outside the timed region; the thread only samples
            import pynvml as nv
            nv.nvmlInit()
            self.hd = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = nv.nvmlDeviceGetMaxClockInfo(self.hd, nv.NVML_CLOCK_SM)
            self.nv = nv
        except Exception:
            self.nv = None
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        if self.nv is not None:                # ~5 ms cadence: dozens of samples inside a 0.2 s timed region
            nv = self.nv
            bits = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))
            while not self.stop_flag:
                try:
                    sm = nv.nvmlDeviceGetClockInfo(self.hd, nv.NVML_CLOCK_SM)
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.hd)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.hd)
                    self.rows.append([str(sm), str(self.mx), "", *("Active" if r & b else "Not Active" for _, b in bits)])
                except Exception:
                    pass
                time.sleep(0.005)
            return
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.th.join(timeout=6)

    def summary(self):
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def dist_setup(n):
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world > 1:
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, local, world


def workload_config(world, B):
    return {"workload": "CIFAR-10 UNet (configs/cifar10.json, 35.7M params, drop 0.1 active) training step: repack + q_sample + fwd + MSE + bwd"
                        + (" + NCCL all-reduce(mean) of the flat fp32 grads, overlapped with the backward chunk by chunk" if world > 1 else ""),
            "per_gpu_batch": B, "global_batch": B * world, "resolution": "3x32x32", "parallelism": f"dp{world}",
            "l2": "4 rotating input batches; activations (2.2 GB fwd) exceed the 126 MB L2"}


def dump_outputs(out_dir, model, losses, n_grad_sample=1 << 22):
    """Write what the timed training step hands its caller after its last step, so that two builds can be compared output
    for output: `losses.npy` (per-sample MSE, float32), `grad_norms.npy` (L2 norm of every parameter's gradient in
    state_dict order, float64) and `grad_sample.npy` (float32 gradient entries at 2^22 fixed positions of the concatenated
    parameter gradients, drawn with seed 0: all 35.7M of them would be 143 MB)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    views = model.grad_views()
    flat = torch.cat([v.flatten() for v in views])
    pick = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:n_grad_sample].sort().values
    np.save(os.path.join(out_dir, "losses.npy"), losses.float().cpu().numpy())
    np.save(os.path.join(out_dir, "grad_norms.npy"), torch.stack([v.double().norm() for v in views]).cpu().numpy())
    np.save(os.path.join(out_dir, "grad_sample.npy"), flat[pick.to(flat.device)].float().cpu().numpy())


def reference_cpu_step(bs):
    """-> (step_fn, kind, what).  The reference's own training step on the host CPU: the UNMODIFIED reference (oracle/_ref,
    staged by build()) - ddpm_torch.UNet(**configs/cifar10.json["model"]) in .train() mode (dropout 0.1 active) under
    ddpm_torch.GaussianDiffusion.train_losses(...).mean().backward() - or, if it is not staged, the oracle port."""
    torch.set_num_threads(CPU_THREADS)
    g = torch.Generator().manual_seed(0)
    x0 = torch.randn(bs, 3, 32, 32, generator=g); t = torch.randint(1000, (bs,), generator=g); noise = torch.randn(bs, 3, 32, 32, generator=g)
    from oracle import ref_loader
    if ref_loader.available():
        ddpm_torch, _ = ref_loader.load()
        cfg = ref_loader.config("cifar10")
        torch.manual_seed(1234)
        model = ddpm_torch.UNet(out_channels=3, **cfg["model"]).train()
        dc = cfg["diffusion"]
        diff = ddpm_torch.GaussianDiffusion(ddpm_torch.get_beta_schedule(dc["beta_schedule"], dc["beta_start"], dc["beta_end"], dc["timesteps"]),
                                            dc["model_mean_type"], dc["model_var_type"], dc["loss_type"])

        def step():
            model.zero_grad(set_to_none=True)
            diff.train_losses(model, x0, t, noise).mean().backward()
        return step, "reference", "unmodified tqch/ddpm-torch (oracle/_ref): ddpm_torch.UNet + GaussianDiffusion.train_losses(...).mean().backward(), train mode"
    from oracle import ddpm_ref as R
    cfg = dict(R.CIFAR10_CFG); cfg["drop_rate"] = 0.0
    sd = {k: v.requires_grad_(True) for k, v in R.make_state_dict(cfg, 1234).items()}
    diff = R.RefDiffusion(R.get_beta_schedule("linear", 1e-4, 0.02, 1000), "fixed-large")

    def step():
        for p in sd.values():
            p.grad = None
        diff.train_losses(lambda x, tt: R.unet_forward(sd, cfg, x, tt), x0, t, noise).mean().backward()
    return step, "port", "oracle port of the reference path (oracle/_ref not staged), dropout 0"


def run_reference(args):
    """The reference's own implementation of the step on the host CPU, all the host threads it can use, at the SAME
    configuration as the main arm (bs=128 per step, cifar10.json as is)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    bs = args.bs
    step, kind, what = reference_cpu_step(bs)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    v = bs / dt
    line = {"impl": "reference", "metric": "unet_train_step_images_per_sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus, bs),
            "cpu_baseline": {"value": v, "unit": "images/s", "cores": CPU_THREADS, "kind": kind,
                             "sample": f"{args.steps} steps of bs={bs}, fp32, torch CPU, {torch.get_num_threads()} threads; {what}"},
            "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    args.emit(line)


def cpu_baseline_sample(bs=128, budget_s=20.0):
    step, kind, what = reference_cpu_step(bs)
    step()
    n, t0 = 0, time.perf_counter()
    while time.perf_counter() - t0 < budget_s and n < 40:
        step(); n += 1
    dt = (time.perf_counter() - t0) / max(n, 1)
    return {"value": bs / dt, "unit": "images/s", "cores": CPU_THREADS, "kind": kind,
            "sample": f"{n} steps of bs={bs} fwd+bwd, fp32, torch CPU, {torch.get_num_threads()} threads; {what}"}


def stock_cuda_reference(dev, my_train_ms, my_sampler_ms, bs=128, sbs=256):
    """north_star's '>=10x the reference's stock torch-CUDA UNet step' denominator: the UNMODIFIED reference modules on this
    same B200 with the reference's settings (fp32 params, TF32 convs, cudnn.benchmark=True as train.py:227-228), and under
    torch.autocast(bf16) for a like-for-like precision; plus its p_sample_step at bs=256."""
    from oracle import ref_loader
    if not ref_loader.available():
        return {"unavailable": "oracle/_ref not staged"}
    ddpm_torch, _ = ref_loader.load()
    cfg = ref_loader.config("cifar10")
    torch.backends.cudnn.benchmark = True
    torch.manual_seed(1234)
    model = ddpm_torch.UNet(out_channels=3, **cfg["model"]).to(dev).train()
    dc = cfg["diffusion"]
    diff = ddpm_torch.GaussianDiffusion(ddpm_torch.get_beta_schedule(dc["beta_schedule"], dc["beta_start"], dc["beta_end"], dc["timesteps"]),
                                        dc["model_mean_type"], dc["model_var_type"], dc["loss_type"])
    g = torch.Generator(device=dev).manual_seed(0)
    x0 = torch.randn(bs, 3, 32, 32, device=dev, generator=g); t = torch.randint(1000, (bs,), device=dev, generator=g)
    nz = torch.randn(bs, 3, 32, 32, device=dev, generator=g)

    def timeit(fn, warm=3, it=8):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        for _ in range(it):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / it

    def step(ac):
        model.zero_grad(set_to_none=True)
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=ac):
            loss = diff.train_losses(model, x0, t, nz).mean()
        loss.backward()
    out = {"kind": "reference", "what": "unmodified ddpm_torch.UNet/GaussianDiffusion on the same GPU, cudnn.benchmark, train mode", "bs": bs}
    out["train_ms_tf32_default"] = timeit(lambda: step(False))
    out["train_ms_bf16_autocast"] = timeit(lambda: step(True))
    out["train_speedup_vs_tf32_default"] = out["train_ms_tf32_default"] / my_train_ms
    out["train_speedup_vs_bf16_autocast"] = out["train_ms_bf16_autocast"] / my_train_ms
    model.eval()
    xs = torch.randn(sbs, 3, 32, 32, device=dev, generator=g)
    tt = torch.full((sbs,), 500, dtype=torch.int64, device=dev)
    with torch.inference_mode():
        out["sampler_step_ms_bs256"] = timeit(lambda: diff.p_sample_step(model, xs, tt), warm=3, it=8)
    if my_sampler_ms:
        out["sampler_step_speedup"] = out["sampler_step_ms_bs256"] / my_sampler_ms
    torch.backends.cudnn.benchmark = False
    del model
    torch.cuda.empty_cache()
    return out


def dominant_kernel_roofline(pk, iters=30):
    """Time the dominant tcgen05 launch of the step in isolation, live, with CUDA events on the launching stream:
    3x3 conv Ci=Co=128 at 32x32, batch 128 (conv3x3_halo2_kernel<128,0>, the CTA-pair kernel; 7 forward + 7 dgrad launches per step share this
    shape, 17% of the step's FLOPs).  Inputs (33.5 MB in + 33.5 MB out per launch) rotate over 8 buffer pairs
    (537 MB > 126 MB L2).  achieved = 2*B*H*W*Co*9*Ci FLOPs / mean launch time."""
    import ctypes as C
    from ddpm_torch_b200 import _lib
    B, H, W, Ci, Co = 128, 32, 32, 128, 128
    nbuf = 8
    xs = [torch.randn(B, H, W, Ci, device="cuda").to(torch.bfloat16) for _ in range(nbuf)]
    ys = [torch.empty(B, H, W, Co, device="cuda", dtype=torch.bfloat16) for _ in range(nbuf)]
    w = (torch.randn(Co, 9 * Ci, device="cuda") * 0.03).to(torch.bfloat16)
    bias = torch.zeros(Co, device="cuda")
    descs = []
    for i in range(nbuf):
        d = _lib.HaloDesc()
        d.NB, d.H, d.W, d.Cout = B, H, W, Co
        d.a_ptr[0] = xs[i].data_ptr(); d.a_C[0] = Ci; d.a_ld[0] = Ci
        d.nseg = 1; d.seg_map[0] = 0; d.seg_taps[0] = 9; d.seg_kchunks[0] = Ci // 64
        d.w = w.data_ptr(); d.ldw = 9 * Ci; d.Ktot = 9 * Ci; d.out = ys[i].data_ptr(); d.bias = bias.data_ptr()
        descs.append(d)
    L = _lib.lib()
    st = _lib.stream_ptr()
    for i in range(nbuf):
        _lib.check(L.ddpm_conv_halo_run(C.byref(descs[i]), st))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for i in range(iters):
        L.ddpm_conv_halo_run(C.byref(descs[i % nbuf]), st)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    flops = 2.0 * B * H * W * Co * 9 * Ci
    ach = flops / (ms * 1e-3) / 1e12
    # traffic: dram__bytes_read.sum + dram__bytes_write.sum of this kernel and shape from the committed ncu --set full capture
    # (profiles/r02_ncu_full_conv3x3_halo2.txt, first launch): 34.01 MB read + 0.40 MB written per launch; algorithmic bytes are
    # 33.5 MB in + 33.5 MB out + 0.3 MB weights (the output is still resident in the 126 MB L2 when the kernel ends)
    return {"bound": "tensor", "achieved": ach, "peak": pk["burst"], "unit": "TFLOP/s", "frac": ach / pk["burst"], "traffic": 34.41e6,
            "kernel": "conv3x3_halo2_kernel<128,0> (cta_group::2 pair): conv3x3 128->128 @32x32 B=128 (isolated, rotating buffers > L2)",
            "ms_per_launch": ms, "gflop_per_launch": flops / 1e9, "peak_source": f"{pk['src']} bf16 burst (MEASURED_PEAKS.json)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bs", type=int, default=128, help="per-GPU batch (weak scaling)")
    ap.add_argument("--no-sampler", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-hq", action="store_true")
    ap.add_argument("--no-stock", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's losses and gradients to DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 training step")
    args.warmup = max(args.warmup, 3)
    # stdout carries exactly ONE JSON line: anything a library writes to fd 1 meanwhile (e.g. the NCCL version banner) goes to stderr
    sys.stdout.flush()
    _real_stdout = os.dup(1); os.dup2(2, 1)
    def emit(obj):
        sys.stdout.flush(); os.dup2(_real_stdout, 1)
        print(json.dumps(obj), flush=True)
    args.emit = emit
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    import ddpm_torch_b200 as D
    from ddpm_torch_b200 import _lib
    rank, local, world = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    _lib.runtime_check()
    pk = peaks()
    torch.manual_seed(1234 + rank)
    B = args.bs
    model = D.UNet(**CIFAR).to(dev).train()
    # non-degenerate weights (the reference init zeroes the last conv of every block -> all-zero gradients upstream)
    with torch.no_grad():
        gi = torch.Generator(device=dev).manual_seed(7)
        for n_, p in model.named_parameters():
            if p.ndim >= 2:
                fan_in = p[0].numel()
                p.copy_((torch.rand(p.shape, device=dev, generator=gi) * 2 - 1) * (3.0 / fan_in) ** 0.5)
    diff = D.GaussianDiffusion(D.get_beta_schedule("linear", 1e-4, 0.02, 1000), "eps", "fixed-large", "mse")
    g = torch.Generator(device=dev).manual_seed(100 + rank)
    # device-resident inputs for `value`: several batches so that consecutive steps do not re-read the same lines
    nb = 4
    x0s = [torch.rand(B, 3, 32, 32, device=dev, generator=g) * 2 - 1 for _ in range(nb)]
    ts = [torch.randint(1000, (B,), device=dev, generator=g) for _ in range(nb)]
    nzs = [torch.randn(B, 3, 32, 32, device=dev, generator=g) for _ in range(nb)]
    L = _lib.lib()
    h = model.prepare(B, 32, 32, training=True)
    ta, tsb = diff._dev_tables(dev)
    losses = torch.empty(B, device=dev)
    gscale = torch.full((B,), 1.0 / B, device=dev)
    stream = torch.cuda.current_stream()

    def step(i):
        sp = _lib.stream_ptr()
        _lib.check(L.ddpm_unet_repack(h, sp))
        k = i % nb
        _lib.check(L.ddpm_train_forward(h, x0s[k].data_ptr(), ts[k].data_ptr(), nzs[k].data_ptr(), ta.data_ptr(), tsb.data_ptr(),
                                        losses.data_ptr(), 1000 + i, sp))
        _lib.check(L.ddpm_train_backward(h, gscale.data_ptr(), sp))
        if world > 1:
            D.parallel.allreduce_grads_overlapped_(model)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    with ClockSampler(local) as cs:
        barrier()
        e0.record()
        for i in range(args.steps):
            step(i)
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1) / args.steps
    clocks = cs.summary()
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = tms.item()
    value = world * B / (ms * 1e-3)
    assert L.ddpm_device_error_flag() == 0
    if args.dump_outputs and rank == 0:                 # before the legs below overwrite the loss and gradient buffers
        dump_outputs(args.dump_outputs, model, losses)
    nf, nbw, npk = (__import__("ctypes").c_int() for _ in range(3))
    import ctypes as C
    L.ddpm_unet_launch_counts(h, C.byref(nf), C.byref(nbw), C.byref(npk))
    launches_per_step = nf.value + nbw.value + npk.value + 3      # + q_sample, mse, mse_grad

    # ---- e2e: public API, batch from pinned host memory, loss read back (+ all-reduce through the same flat buffer)
    host_x = [torch.empty(B, 3, 32, 32).uniform_(-1, 1).pin_memory() for _ in range(nb)]
    gen = torch.Generator(device=dev).manual_seed(8191 + rank)

    def e2e_step(i):
        x = host_x[i % nb].to(dev, non_blocking=True)
        t = torch.randint(1000, (B,), device=dev, generator=gen)
        nz = torch.randn(B, 3, 32, 32, device=dev, generator=gen)
        model.zero_grad(set_to_none=True)
        loss = diff.train_losses(model, x, t, nz).mean()
        loss.backward()
        if world > 1:
            D.parallel.allreduce_grads_overlapped_(model)
        return loss.item()

    for i in range(args.warmup):
        e2e_step(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        e2e_step(i)
    e1.record()
    barrier()
    ems = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_val = world * B / (ems.item() * 1e-3)

    # ---- SURVEY 8d config 2 "with and without optimiser/EMA": the same device-resident step followed by the fused
    # clip_grad_norm + Adam + LR warm-up + EMA update (ddpm_opt_step, 2 launches over the flat fp32 buffers)
    from ddpm_torch_b200.optim import EMA, FusedAdam, hbm_bytes_per_step
    opt = FusedAdam(model, lr=2e-4, betas=(0.9, 0.999), warmup=5000, grad_norm=1.0, ema=EMA(model, 0.9999))

    def step_opt(i):
        step(i)
        opt.step()

    for i in range(args.warmup):
        step_opt(i)
    barrier()
    e0.record()
    for i in range(args.steps):
        step_opt(i)
    e1.record()
    barrier()
    oms = torch.tensor([e0.elapsed_time(e1) / args.steps], device=dev)
    if world > 1:
        dist.all_reduce(oms, op=dist.ReduceOp.MAX)
    torch.cuda.synchronize()
    e0.record()
    for i in range(20):
        opt.step()
    e1.record()
    torch.cuda.synchronize()
    opt_ms = e0.elapsed_time(e1) / 20
    n_par = model.flat_params.numel()
    opt_gbs = hbm_bytes_per_step(n_par, ema=True) / (opt_ms * 1e-3) / 1e9
    with_opt = {"value": world * B / (oms.item() * 1e-3), "unit": "images/s", "ms_per_step": oms.item(),
                "what": "step + fused clip_grad_norm/Adam/LR-warm-up/EMA (utils/train.py:159-165) over the flat buffers",
                "opt_ms_isolated": opt_ms, "launches": 2,
                "roofline": {"bound": "hbm", "achieved": opt_gbs, "peak": pk["hbm"], "unit": "GB/s",
                             "frac": opt_gbs / pk["hbm"],
                             "algorithmic_bytes": hbm_bytes_per_step(n_par, ema=True), "traffic": None}}

    line = {"metric": "unet_train_step_images_per_sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": workload_config(world, B),
            "e2e": {"value": e2e_val, "unit": "images/s", "h2d_bytes_per_step": B * 3 * 32 * 32 * 4, "d2h_bytes_per_step": 4,
                    "ms_per_step": ems.item(), "api": "GaussianDiffusion.train_losses(model, x, t, noise).mean().backward()"},
            "with_optimizer": with_opt,
            "gpu_launches": launches_per_step * args.steps, "launches_per_step": launches_per_step, "clocks": clocks,
            "step_tflops": world * B * TRAIN_GFLOP_PER_IMG / ms, "step_frac_of_sustained_peak": B * TRAIN_GFLOP_PER_IMG / ms / pk["sustained"]}

    def maxr(v):
        tv = torch.tensor([v], device=dev)
        if world > 1:
            dist.all_reduce(tv, op=dist.ReduceOp.MAX)
        return tv.item()

    extras = {}
    if not args.no_sampler:
        extras["sampler"] = bench_sampler(D, model, dev, rank, world, barrier, maxr, pk)
    del opt
    if not args.no_hq:
        model = None
        torch.cuda.empty_cache()
        extras.update(bench_hq(D, _lib, dev, rank, world, barrier, maxr, pk))
    if rank == 0:
        line.update(extras)
        line["roofline"] = dominant_kernel_roofline(pk)
        if world == 1 and not args.no_stock:
            try:
                line["vs_stock_cuda"] = stock_cuda_reference(dev, ms, (extras.get("sampler") or {}).get("ddim50", {}).get("ms_per_step"))
            except Exception as e:                      # informational leg: never costs the headline line
                line["vs_stock_cuda"] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_sample(B)
        args.emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def bench_sampler(D, model, dev, rank, world, barrier, maxr, pk, bs=256):
    """config 3: p_sample T=1000 (fixed-large) and DDIM S=50 (eta 0), bs=256 PER GPU (images sharded by rank,
    generate.py:105-110 rule, different seed per rank, no collective), one CUDA-graph replay per timestep."""
    out = {"per_gpu_batch": bs, "global_batch": D.parallel.shard_size(bs * world, rank, world) * world, "sharding": "by image, no collective"}
    betas = D.get_beta_schedule("linear", 1e-4, 0.02, 1000)
    model.eval()
    base = D.GaussianDiffusion(betas, "eps", "fixed-large", "mse")
    ddim = D.DDIM.from_ddpm(D.GaussianDiffusion(betas, "eps", "fixed-small", "mse"), eta=0.0, subsequence=D.get_selection_schedule("linear", 50, 1000))
    n_img = D.parallel.shard_size(bs * world, rank, world)
    x = None
    for name, d, S in (("ddim50", ddim, 50), ("ancestral1000", base, 1000)):
        if name == "ddim50":
            d.p_sample(model, shape=(n_img, 3, 32, 32), device=dev, seed=1 + rank)      # warm-up (plan, graph)
        barrier()
        e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
        e0.record()
        x = d.p_sample(model, shape=(n_img, 3, 32, 32), device=dev, seed=2 + rank)
        e1.record()
        barrier()
        s = maxr(e0.elapsed_time(e1)) * 1e-3
        assert torch.isfinite(x).all()
        tf = n_img * FWD_GFLOP_PER_IMG * S / s / 1e3
        out[name] = {"images_per_s": world * n_img / s, "seconds_per_batch": s, "ms_per_step": s / S * 1e3, "steps": S,
                     "tflops_per_gpu": tf, "frac_of_burst_peak": tf / pk["burst"], "frac_of_sustained_peak": tf / pk["sustained"],
                     "rng": "torch generator (reference-compatible stream)"}
    if rank == 0 and world == 1:
        # generate.py:128-130 tail: device uint8 NHWC conversion + pinned async D2H of the finished batch vs the reference's
        # fp32 .cpu() + five host passes
        from ddpm_torch_b200.postprocess import to_uint8_host_async
        from oracle import ddpm_ref as R
        pinned, ev = to_uint8_host_async(x); ev.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            pinned, ev = to_uint8_host_async(x, pinned); ev.synchronize()
        t_dev = (time.perf_counter() - t0) / 10
        t0 = time.perf_counter()
        for _ in range(3):
            ref = R.to_uint8_nhwc(x.cpu()).numpy()
        t_ref = (time.perf_counter() - t0) / 3
        assert (ref == pinned.numpy()).all()
        out["postprocess_uint8"] = {"device_kernel_plus_pinned_d2h_ms": t_dev * 1e3, "reference_host_path_ms": t_ref * 1e3, "bs": bs,
                                    "bit_exact_vs_reference_expression": True}
    model.train()
    return out


def bench_hq(D, _lib, dev, rank, world, barrier, maxr, pk, train_bs=4, sample_bs=8, steps=10, warmup=3):
    """BASELINE configs 4 and 5 (configs/celebahq.json, 113.7M parameters, 3x256x256): training step at 4 images per GPU with
    the NCCL mean all-reduce of the 455 MB flat fp32 gradient, and DDIM S=100 (eta 0) at 8 images per GPU (sharded by image,
    no collective).  Weak scaling in N, like the headline."""
    L = _lib.lib()
    torch.manual_seed(4321 + rank)
    model = D.UNet(**HQ).to(dev).train()
    with torch.no_grad():
        gi = torch.Generator(device=dev).manual_seed(7)
        for _, p in model.named_parameters():
            if p.ndim >= 2:
                p.copy_((torch.rand(p.shape, device=dev, generator=gi) * 2 - 1) * (3.0 / p[0].numel()) ** 0.5)
    betas = D.get_beta_schedule("linear", 1e-4, 0.02, 1000)
    diff = D.GaussianDiffusion(betas, "eps", "fixed-small", "mse")
    g = torch.Generator(device=dev).manual_seed(200 + rank)
    B = train_bs
    x0 = torch.rand(B, 3, 256, 256, device=dev, generator=g) * 2 - 1
    t = torch.randint(1000, (B,), device=dev, generator=g); nz = torch.randn(B, 3, 256, 256, device=dev, generator=g)
    h = model.prepare(B, 256, 256, training=True)
    ta, tsb = diff._dev_tables(dev); losses = torch.empty(B, device=dev); gs = torch.full((B,), 1.0 / B, device=dev)

    def step(i):
        sp = _lib.stream_ptr()
        _lib.check(L.ddpm_unet_repack(h, sp))
        _lib.check(L.ddpm_train_forward(h, x0.data_ptr(), t.data_ptr(), nz.data_ptr(), ta.data_ptr(), tsb.data_ptr(), losses.data_ptr(), 0, sp))
        _lib.check(L.ddpm_train_backward(h, gs.data_ptr(), sp))
        if world > 1:
            D.parallel.allreduce_grads_overlapped_(model)
    for i in range(warmup):
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(True), torch.cuda.Event(True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    barrier()
    ms = maxr(e0.elapsed_time(e1) / steps)
    assert torch.isfinite(losses).all() and L.ddpm_device_error_flag() == 0
    tf = B * 3 * HQ_FWD_GFLOP_PER_IMG / ms
    out = {"hq_train": {"images_per_s": world * B / (ms * 1e-3), "ms_per_step": ms, "per_gpu_batch": B, "global_batch": B * world,
                        "tflops_per_gpu": tf, "frac_of_burst_peak": tf / pk["burst"], "frac_of_sustained_peak": tf / pk["sustained"],
                        "allreduce_bytes": model.flat_grads.numel() * 4 if world > 1 else 0, "steps": steps,
                        "what": "celebahq.json UNet (113.7M params) 3x256x256: repack + q_sample + fwd + MSE + bwd" + (" + NCCL all-reduce(mean)" if world > 1 else "")}}
    # ---- config 5: DDIM-100 at 8 images per GPU
    model._ws = None; model._plan_key = None; model._grads = None
    torch.cuda.empty_cache()
    model.eval()
    ddim = D.DDIM.from_ddpm(diff, eta=0.0, subsequence=D.get_selection_schedule("linear", 100, 1000))
    n_img = D.parallel.shard_size(sample_bs * world, rank, world)
    ddim.p_sample(model, shape=(n_img, 3, 256, 256), device=dev, seed=3 + rank)        # warm-up (plan, step graph)
    barrier()
    e0.record()
    x = ddim.p_sample(model, shape=(n_img, 3, 256, 256), device=dev, seed=5 + rank)
    e1.record()
    barrier()
    s = maxr(e0.elapsed_time(e1)) * 1e-3
    assert torch.isfinite(x).all() and L.ddpm_device_error_flag() == 0
    tf = n_img * HQ_FWD_GFLOP_PER_IMG * 100 / s / 1e3
    out["hq_ddim100"] = {"images_per_s": world * n_img / s, "seconds_per_batch": s, "ms_per_step": s * 10.0, "per_gpu_batch": n_img,
                         "global_batch": n_img * world, "steps": 100, "tflops_per_gpu": tf, "frac_of_burst_peak": tf / pk["burst"],
                         "frac_of_sustained_peak": tf / pk["sustained"], "sharding": "by image (generate.py:105-110), no collective"}
    return out


if __name__ == "__main__":
    main()
