#!/usr/bin/env python
"""Benchmark of the hot path: SD1.5 LoRA (rank 8, every attn1/attn2 Linear) training step, 512x512 (64x64 latents),
batch 4 per GPU, bf16 kernels / fp32 master weights -- BASELINE.json `configs[1]`, metric "LoRA-train images/sec".

  python bench.py [--gpus N] [--steps K] [--warmup W]            product arm (B200 kernels): K timed steps with inputs resident,
                  [--dump-outputs DIR]                           then K timed steps fed from pinned host memory; DIR receives what
                                                                 the last step left (see dump_outputs)
  python bench.py --impl reference [--gpus N] ...                CPU arm: the oracle restatement of the reference path
                                                                 (diffusers UNet semantics + hcpdiff LoRA operator + train_ac
                                                                 step order) on the host cores -- the reference itself cannot
                                                                 run here (diffusers/accelerate/hydra are not installable)
For N > 1 launch with torchrun (one rank per GPU); rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

F_FWD = 803.27e9                 # algorithmic FLOP per image, forward (BASELINE.md section 3 / SURVEY.md App. B)
F_ATTN = 126.05e9
F_STEP = 2 * F_FWD + F_ATTN      # LoRA training step with frozen base: 1732.6 GFLOP / image
METRIC = "LoRA-train images/sec SD1.5 512px"
PER_GPU_BATCH = 4
LORA_RANK = 8


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1423.3), d.get("bf16_tflops", 1713.4), d.get("hbm_gbs", 6567.7), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


def usable_cores() -> int:
    """Host threads this process may really use: the scheduler affinity mask capped by the cgroup CPU quota (a box that
    shows 128 logical CPUs but grants a 16-CPU quota thrashes with 128 threads)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except (OSError, ValueError):
        pass
    return n


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); smax.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference path)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(max_steps: int, warmup: int, budget_s: float, batch: int = 1):
    """One step = `batch` images (64x64 latents, 77 tokens) through the reference step order (train_ac.py:467-504): forward ->
    MSE(eps) -> backward -> clip 1.0 -> AdamW -> zero_grad, fp32, all host threads.  Steps stop early when `budget_s` is spent."""
    from oracle import unet_ref as U
    cores = usable_cores()
    torch.set_num_threads(cores)
    spec = U.SD15
    sd = U.init_params(spec)
    lora = U.init_lora(spec, rank=LORA_RANK, up_std=0.0)
    params = []
    for blocks in lora.values():
        for e in blocks:
            e.W_down.requires_grad_(True)
            e.W_up.requires_grad_(True)
            params += [e.W_down, e.W_up]
    opt = torch.optim.AdamW(params, lr=1e-4, weight_decay=1e-2)
    acp = U.ddpm_alphas_cumprod()
    lat, noise, t, ehs = U.synthetic_batch(batch, spec, seed=1234)

    def one_step():
        x_t = U.add_noise(lat, noise, t, acp)
        pred = U.unet_forward(sd, x_t, t, ehs, lora=lora, spec=spec)
        loss = torch.nn.functional.mse_loss(pred.float(), noise.float(), reduction="none").mean()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        opt.zero_grad(set_to_none=False)
        return float(loss.detach())

    t_start = time.perf_counter()
    done_w = 0
    for _ in range(warmup):
        one_step()
        done_w += 1
        if time.perf_counter() - t_start > budget_s * 0.4:
            break
    t0 = time.perf_counter()
    done = 0
    while done < max_steps:
        one_step()
        done += 1
        if time.perf_counter() - t_start > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"images_per_s": done * batch / dt, "steps_run": done, "warmup_run": done_w, "seconds": dt, "cores": cores, "batch": batch}


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    # the product arm's configuration: batch 4 per step (a step takes ~20 s on 16 host cores: the run is time-bounded, `steps` says
    # how many were timed)
    r = cpu_reference_steps(args.steps, min(args.warmup, 1), budget_s=210.0, batch=PER_GPU_BATCH)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["images_per_s"], "unit": "images/s", "n_gpus": args.gpus, "steps": r["steps_run"],
        "requested_steps": args.steps, "warmup": r["warmup_run"], "ms_per_step": 1e3 * r["seconds"] / r["steps_run"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SD1.5 UNet LoRA r=8 on all attn1/attn2 Linear (128 layers), bs=4, 512x512 (64x64 latent), 77 tokens; "
                               "step = add_noise + UNet fwd + MSE + bwd + clip + AdamW",
                   "per_step_sample": f"{r['batch']} images (the product arm's per-GPU batch): fwd + MSE + bwd + clip + AdamW",
                   "global_batch": r["batch"], "per_gpu_batch": r["batch"], "lora_rank": LORA_RANK},
        "cpu_baseline": {"value": r["images_per_s"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                         "sample": f"{r['steps_run']} timed step(s) of {r['batch']} images each after {r['warmup_run']} warm-up; oracle/unet_ref.py "
                                   "(restated diffusers UNet + reference LoRA operator), torch CPU fp32, time-bounded"},
        "e2e": {"value": r["images_per_s"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------------
# product arm
# ----------------------------------------------------------------------------------------------------------------------
def time_kernel(fn, iters=10):
    for _ in range(2):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def ncu_dram_traffic(summary=None):
    """DRAM bytes (read + write) of ONE launch of the dominant kernel, from the committed `ncu --set full` summary of the same
    kernel at the same shape (attention backward, B=4 H=8 L=4096 d=40).  None when the file is absent."""
    import csv
    here = os.path.dirname(os.path.abspath(__file__))
    if summary is None:          # the newest committed capture of the kernel
        summary = next((n for n in ("profiles/r02_ncu_attn_bwd.summary.csv", "profiles/r01_ncu_attn_bwd_v23.summary.csv")
                        if os.path.exists(os.path.join(here, n))), "profiles/r01_ncu_attn_bwd_v23.summary.csv")
    path = os.path.join(here, summary)
    try:
        rows = list(csv.reader(open(path)))
        hdr, unit, val = rows[0], rows[1], rows[2]
        scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        tot = 0.0
        for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            i = hdr.index(name)
            tot += float(val[i]) * scale[unit[i]]
        return {"bytes_per_launch": tot, "kernel": "attn_bwd_kernel B4 H8 L4096 d40", "source": summary}
    except (OSError, ValueError, KeyError, IndexError):
        return None


def dominant_kernel_roofline(peak_tflops):
    """Live CUDA-event timing of the kernels that dominate the step, at their benchmark shapes (B=4)."""
    from hcp_diffusion_b200 import ops
    B, H, L, d = PER_GPU_BATCH, 8, 4096, 40
    C = H * d
    qkv = torch.randn(B, L, 3 * C, device="cuda").to(torch.bfloat16).requires_grad_(True)
    o = ops.attention(H, C, (0, C, 2 * C), qkv)
    do = torch.randn_like(o)
    ms_f = time_kernel(lambda: ops.attention(H, C, (0, C, 2 * C), qkv.detach()))

    def bwd():
        oo = ops.attention(H, C, (0, C, 2 * C), qkv)
        oo.backward(do)
    ms_fb = time_kernel(bwd)
    ms_b = ms_fb - ms_f
    fl_f = 4.0 * B * H * L * L * d
    fl_b = 10.0 * B * H * L * L * d
    out = {
        "attn_fwd_L4096_d40": {"ms": ms_f, "tflops": fl_f / ms_f * 1e-9, "frac": fl_f / ms_f * 1e-9 / peak_tflops},
        "attn_bwd_L4096_d40": {"ms": ms_b, "tflops": fl_b / ms_b * 1e-9, "frac": fl_b / ms_b * 1e-9 / peak_tflops},
    }
    x = torch.randn(B, 4096, 320, device="cuda").to(torch.bfloat16)
    w = torch.randn(320, 320, 3, 3, device="cuda") * 0.02
    pack = ops.ConvPack(w, None, 1)
    ms_c = time_kernel(lambda: ops.conv3x3(pack, x, (B, 64, 64)))
    fl_c = 2.0 * B * 4096 * 320 * 9 * 320
    out["conv3x3_320_320_64x64"] = {"ms": ms_c, "tflops": fl_c / ms_c * 1e-9, "frac": fl_c / ms_c * 1e-9 / peak_tflops}
    return out


def count_step_flops(step, host):
    """Algorithmic FLOP of ONE training step, summed over the C-ABI GEMM / convolution / attention calls it makes (2 M N K per GEMM
    segment, 2 M Cout 9 Cin per convolution, 4 / 10 B H Lq Lkv d per attention forward / backward).  Used for workloads without a
    published per-image figure (config 4); the LoRA-gradient kernels are not counted.  The calls are logged while the step's CUDA graph
    is captured, nothing is timed here."""
    import hcp_diffusion_b200.engine as _eng
    import hcp_diffusion_b200.ops as _ops
    from hcp_diffusion_b200 import _lib
    total = [0.0]
    orig = _lib.call

    def logged(name, *a):
        try:
            o = a[0]._obj if a and hasattr(a[0], "_obj") else None
            if name == "hcp_gemm_bf16":
                total[0] += 2.0 * o.M * o.N * sum(o.k[i] for i in range(o.nseg))
            elif name == "hcp_conv3x3_bf16":
                s_ = o.stride
                mo = o.B * (o.Hin // s_) * (o.Win // s_) if o.mode == 0 else o.B * o.Hin * o.Win     # mode 1: dY pixels of the stride-2 dgrad
                total[0] += 2.0 * mo * o.Cout * 9 * o.Cin
            elif name == "hcp_attn_fwd_bf16":
                total[0] += 4.0 * o.B * o.H * o.Lq * o.Lkv * o.d
            elif name == "hcp_attn_bwd_bf16":
                total[0] += 10.0 * o.B * o.H * o.Lq * o.Lkv * o.d
        except Exception:      # noqa: BLE001  (a logging helper must never break the run)
            pass
        return orig(name, *a)

    _lib.call = _ops.call = _eng.call = logged
    try:
        step.step(*host)                               # first call: warm-up + CUDA-graph capture; every launch goes through `call` once per pass
    finally:
        _lib.call = _ops.call = _eng.call = orig
    # the capture path runs the step three times (two warm-up passes + the capture): FLOP of one pass
    return total[0] / 3.0


def attn_tensor_pipe_pct():
    """BASELINE.json's second metric, "attn tensor-pipe % of peak": sm__pipe_tensor... pct of peak of the attention kernels at the
    benchmark shape (B=4, H=8, L=4096, d=40), read from the committed `ncu --set full` summaries (a number taken under a profiler is
    never a bench value: this is evidence attached to the line, not something measured by this run)."""
    import csv
    out = {}
    for key, names in (("fwd", ("profiles/r02_ncu_attn_fwd.summary.csv", "profiles/r01_ncu_attn_fwd_v23.summary.csv")),
                       ("bwd", ("profiles/r02_ncu_attn_bwd.summary.csv", "profiles/r01_ncu_attn_bwd_v23.summary.csv"))):
        for name in names:
            path = os.path.join(ROOT, name)
            try:
                rows = list(csv.reader(open(path)))
                hdr, val = rows[0], rows[2]
                # the SM-average over the kernel's whole duration (not the busiest SM, not "while active")
                pref = "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed"
                cols = [i for i, h in enumerate(hdr) if h == pref] or \
                       [i for i, h in enumerate(hdr) if h.startswith("sm__pipe_tensor") and "avg.pct_of_peak_sustained_elapsed" in h]
                if cols:
                    out[key] = {"pct": float(val[cols[0]]), "metric": hdr[cols[0]], "source": name}
                    break
            except (OSError, ValueError, IndexError):
                continue
    return out or None


DUMP_MAX_PARAMS = 8 << 20        # float32 elements (32 MB): a larger parameter buffer is dumped as a fixed, seeded sample


def dump_outputs(out_dir, step):
    """What a caller of the training step holds after the last timed step: that step's loss (loss.npy, shape [1]) and the trainable
    parameters AdamW left (params.npy: the flat fp32 parameter buffer, or DUMP_MAX_PARAMS elements of it at sorted indices drawn with
    seed 0 when it is larger, e.g. the 860M parameters of --config 3).  Same arguments -> same inputs and step count, so the files of
    two builds can be compared element for element.  They agree to a tolerance, not bitwise: the kernels' fp32 atomic accumulation
    order varies, and two runs of one build on a B200 (1000 W) differed by 2e-5 (relative) in loss and 2e-3 relative L2 in the
    parameters with --warmup 5 --steps 20."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    params = step.flat.data
    if params.numel() > DUMP_MAX_PARAMS:
        idx = torch.randint(0, params.numel(), (DUMP_MAX_PARAMS,), generator=torch.Generator().manual_seed(0)).sort().values
        params = params[idx.to(params.device)]
    np.save(os.path.join(out_dir, "loss.npy"), step.loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "params.npy"), params.detach().float().cpu().numpy())


def run_product_arm(args, rank, world, local_rank):
    import torch.distributed as dist
    from hcp_diffusion_b200 import _lib
    from hcp_diffusion_b200.engine import LoraTrainStep
    from hcp_diffusion_b200.models import UNet2DConditionModel
    from hcp_diffusion_b200.utils.cfg_net_tools import make_hcpdiff
    from oracle import unet_ref as U   # used for the synthetic weight/input generators and the cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.check(_lib.lib().hcp_device_check(), "hcp_device_check")
    sustained, burst, hbm, peak_src = measured_peaks()
    # the adapters draw W_down (kaiming-uniform) from the global generators on the device: seeded, so every run trains the same weights
    torch.manual_seed(0)

    spec = U.SD15
    added = None
    if args.config == 4:
        # BASELINE configs[3]: SDXL-base UNet, LoRA rank 16 on attn + ff Linears and the resnet / sampler convolutions (locon), bs 2 / GPU,
        # 1024x1024 (128x128 latent), 77 x 2048 text tokens + text_time conditioning (reference cfgs/train/examples/locon.yaml shapes)
        with torch.device("meta"):
            unet = UNet2DConditionModel(sample_size=128, block_out_channels=(320, 640, 1280), attention_head_dim=(5, 10, 20), cross_attention_dim=2048,
                                        down_block_types=("DownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D"),
                                        up_block_types=("CrossAttnUpBlock2D", "CrossAttnUpBlock2D", "UpBlock2D"),
                                        transformer_layers_per_block=(1, 2, 10), use_linear_projection=True, addition_embed_type="text_time",
                                        addition_time_embed_dim=256, projection_class_embeddings_input_dim=2816)
        unet = unet.to_empty(device=dev)
        gen = torch.Generator(device=dev).manual_seed(0)
        with torch.no_grad():
            for name, p_ in unet.named_parameters():           # random init (no checkpoints offline): fan-in scaled weights, unit norm scales
                if p_.dim() > 1:
                    p_.normal_(0, p_[0].numel() ** -0.5, generator=gen)
                elif "norm" in name and name.endswith("weight"):
                    p_.fill_(1.0)
                else:
                    p_.zero_()
        unet = unet.requires_grad_(False).eval()
    else:
        unet = UNet2DConditionModel()
        unet.load_state_dict(U.init_params(spec, seed=0))
        unet = unet.to(dev).requires_grad_(False).eval()
    if args.config == 4:
        layers = [r"re:.*\.attn.?$", r"re:.*\.ff$", r"re:.*\.resnets\.\d+\.conv[12]$", r"re:.*\.conv_shortcut$", r"re:.*samplers\.0\.conv$"]
        groups, lora = make_hcpdiff(unet, None, [{"lr": 1e-4, "rank": 16, "alpha": 1.0, "dropout": 0.0, "layers": layers}])
        B, f_step, metric = 2, None, "LoRA-train images/sec SDXL 1024px"
        use_graph = True
        what = "SDXL-base UNet LoRA r=16 on attn + ff Linear and resnet / sampler Conv2d (locon, %d params), bs=2/GPU"
    elif args.config == 3:
        # BASELINE configs[2]: DreamBooth full fine-tune, no LoRA, bs 16 / GPU (reference cfgs/train/examples/DreamBooth.yaml:6-10)
        groups, lora = make_hcpdiff(unet, [{"lr": 1e-6, "layers": [""]}], None)
        B, f_step, metric = 16, 3 * F_FWD, "full fine-tune images/sec SD1.5 512px"
        # N > 1: eager launches so that the 3.4 GB gradient all-reduce is bucketed under the backward pass (HCP_BENCH_EAGER=1 forces the
        # same mode on one GPU: the baseline the exposed all-reduce time of N > 1 is read against)
        use_graph = world == 1 and os.environ.get("HCP_BENCH_EAGER", "0") != "1"
        what = "SD1.5 UNet full fine-tune (every parameter, %d params), bs=16/GPU"
    else:
        groups, lora = make_hcpdiff(unet, None, [{"lr": 1e-4, "rank": LORA_RANK, "alpha": 1.0, "dropout": 0.0, "layers": [r"re:.*\.attn.?$"]}])
        B, f_step, metric = PER_GPU_BATCH, F_STEP, METRIC
        use_graph = True
        what = "SD1.5 UNet LoRA r=8 on all attn1/attn2 Linear (128 layers, %d params), bs=4/GPU"
    n_train = sum(p.numel() for g in groups for p in g["params"])
    step = LoraTrainStep(unet, groups, weight_decay=1e-2, max_grad_norm=1.0, use_cuda_graph=use_graph)
    step.sync_params(0)

    if args.config == 4:
        g = torch.Generator().manual_seed(1234 + rank)
        lat, noise = torch.randn(B, 4, 128, 128, generator=g), torch.randn(B, 4, 128, 128, generator=g)
        t, ehs = torch.randint(0, 1000, (B,), generator=g), torch.randn(B, 77, 2048, generator=g)
        added = {"text_embeds": torch.randn(B, 1280, generator=g).pin_memory(),
                 "time_ids": torch.tensor([[1024.0, 1024.0, 0.0, 0.0, 1024.0, 1024.0]]).repeat(B, 1).pin_memory()}
    else:
        lat, noise, t, ehs = U.synthetic_batch(B, spec, seed=1234 + rank)
    host = [x.pin_memory() for x in (lat, noise, t, ehs)]
    h2d = sum(x.numel() * x.element_size() for x in host) + (sum(v.numel() * v.element_size() for v in added.values()) if added else 0)
    if added is not None:
        host.append(added)
    if f_step is None:
        f_step = count_step_flops(step, host) / B          # algorithmic FLOP of the GEMM / conv / attention calls of one step, per image

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    losses = []

    def e2e_step():
        loss = step.step(*host)
        losses.append(float(loss.cpu()))          # the per-step D2H read of the result (reference: loss.item(), train_ac.py:504)

    dev_in = [({k: v.to(dev) for k, v in x.items()} if isinstance(x, dict) else x.to(dev)) for x in host]

    def resident_step():
        if use_graph:
            step.step_resident()
        else:
            step.step(*dev_in)

    # warm-up (also captures the CUDA graphs)
    for _ in range(max(args.warmup, 3)):
        e2e_step()
    launches0 = _lib.launch_count
    resident_step()
    launches_per_step = (_lib.launch_count - launches0) if not use_graph else step.launches_per_step
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_resident = timed(resident_step, args.steps)
    clocks = sampler.stop()
    ms_e2e = timed(e2e_step, args.steps)
    assert all(l == l and l < 1e4 for l in losses), "loss diverged / NaN"

    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, step)
    imgs = world * B * args.steps
    value = imgs / (ms_resident * 1e-3)
    e2e_value = imgs / (ms_e2e * 1e-3)
    achieved = value / world * f_step * 1e-12
    # the denominator that matches the clocks this run saw: boost clocks for the whole timed region -> the burst peak
    boosted = bool(clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and clocks["sm_mhz"] >= 0.9 * clocks["sm_max_mhz"])
    peak = burst if boosted else sustained
    kern = dominant_kernel_roofline(burst) if (world == 1 and args.config == 2) else None
    res_txt = "1024x1024 (128x128 latent), 77 x 2048 tokens + text_time conditioning" if args.config == 4 else "512x512 (64x64 latent), 77 tokens"
    line = {
        "metric": metric, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_resident / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": (what % n_train) + ", " + res_txt + "; step = add_noise + UNet fwd + MSE + bwd + grad all-reduce + clip + AdamW",
                   "baseline_config": args.config, "global_batch": world * B, "per_gpu_batch": B, "lora_rank": {2: LORA_RANK, 3: 0, 4: 16}[args.config],
                   "parallelism": f"dp{world}",
                   "l2": "working set (1.7 GB bf16 weights + activations) is far larger than the 126 MB L2; no explicit flush",
                   "cuda_graph": use_graph, "grad_checkpointing": False,
                   "side_stream": os.environ.get("HCP_SIDE_STREAM", "1") != "0", "pdl": os.environ.get("HCP_PDL", "1") != "0"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms_e2e / args.steps, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4},
        "gpu_launches": launches_per_step * args.steps,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "frac_vs_burst": achieved / burst, "frac_vs_sustained": achieved / sustained,
                     "traffic": ncu_dram_traffic(),
                     "peak_source": f"{peak_src} {'bf16_tflops (burst: the timed region ran at boost clocks)' if boosted else 'bf16_tflops_sustained'}; "
                                    f"burst {burst}, sustained {sustained}",
                     "flop_per_image": f_step, "kernels": kern, "attn_tensor_pipe_pct": attn_tensor_pipe_pct()},
        "final_loss": losses[-1],
    }
    if world == 1 and not args.no_cpu_baseline and args.config == 2:
        r = cpu_reference_steps(1, 0, budget_s=30.0, batch=PER_GPU_BATCH)
        line["cpu_baseline"] = {"value": r["images_per_s"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                                "sample": "1 training step of 4 images (the benchmark batch, 64x64 latents): oracle/unet_ref.py fp32 on all host "
                                          "threads, no warm-up"}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="hcpb200", choices=["hcpb200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's loss and the trained parameters to DIR/<name>.npy (float32)")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4],
                    help="BASELINE.json config: 2 = SD1.5 LoRA r8 bs 4/GPU (the headline, default); 3 = SD1.5 full fine-tune bs 16/GPU; "
                         "4 = SDXL-base LoRA r16 attn + Conv2d bs 2/GPU, 1024x1024")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the product arm computed; the reference arm has no such output")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus:
        if args.gpus > 1:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # rank 0 prints ONE json line on stdout: NCCL's version banner / debug lines (whatever NCCL_DEBUG the box exports) go to stderr
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_product_arm(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
