#!/usr/bin/env python
"""Benchmark of the vdm4cdm hot path on B200: reverse ancestral sampling with the 128^3 conditional VDM
denoiser (BASELINE.json configs[1]/[4]: chs=[32,64,128,256], conditioning field + 6 parameters).

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU oracle port on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # ... and write the last timed step's outputs to DIR

A "step" is one reverse step of the chain for the whole batch of realisations on every rank: one CUNet
forward (about 30 tcgen05 conv launches + the fused elementwise kernels) plus the fused sampler update.
Realisations are independent units, so N GPUs run N x batch realisations with no collective in the
data path (weak scaling); timing is CUDA events bracketed by a barrier + synchronize, max over ranks.
Rank 0 prints ONE JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "denoiser voxel-steps/s at 128^3 (reverse ancestral sampling)"
UNIT = "voxel-steps/s"
PARAM_LO = [0.1, 0.6, 0.25, 0.25, 0.5, 0.5]      # CAMELS parameter ranges (SURVEY.md section 8d)
PARAM_HI = [0.5, 1.0, 4.0, 4.0, 2.0, 2.0]
DUMP_MAX_ELEMENTS = 1 << 22      # per dumped array (16 MiB of float32): the two arrays of --dump-outputs stay under 64 MB
DUMP_SAMPLE_SEED = 2024


def synthetic_batch(batch, grid, seed, device="cpu"):
    """x = randn, conditioning = 0.7 x + 0.3 randn, 6 parameters uniform in the CAMELS ranges (seed 42 + rank)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((batch, 1, grid, grid, grid), generator=g)
    cond = 0.7 * x + 0.3 * torch.randn((batch, 1, grid, grid, grid), generator=g)
    lo, hi = torch.tensor(PARAM_LO), torch.tensor(PARAM_HI)
    params = lo + (hi - lo) * torch.rand((batch, 6), generator=g)
    return x.to(device), cond.to(device), params.to(device)


def model_kwargs(grid, chs):
    return dict(shape=(1, grid, grid, grid), chs=chs, s_conditioning_channels=1, v_conditioning_dims=[6],
                t_conditioning=True, norm_groups=8, mid_attn=False, dropout_prob=0.1, conv_padding_mode="zeros",
                n_attention_heads=4)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons of one GPU, sampled every 50 ms while the timed region runs."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 7 and r[3 + i].lower().startswith("active") for r in self.rows)]
        busy = [v for v in sm if v > 0.5 * (mx[0] if mx else 1)] or sm
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": mx[0] if mx else None,
                "reasons": reasons, "samples": len(sm)}


def dump_outputs(out_dir, arrays):
    """Write each tensor of ``arrays`` as ``out_dir/<name>.npy`` in float32.  A tensor of at most DUMP_MAX_ELEMENTS
    elements is written whole, in its shape; a larger one as the 1-D array of its elements at DUMP_MAX_ELEMENTS flat
    indices drawn without replacement by numpy's default_rng(DUMP_SAMPLE_SEED) and sorted.  The indices depend on the
    element count only, so two runs with the same arguments can be compared element for element."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_MAX_ELEMENTS:
            idx = np.sort(np.random.default_rng(DUMP_SAMPLE_SEED).choice(t.numel(), DUMP_MAX_ELEMENTS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ---------------------------------------------------------------------------------------------------------
def cpu_oracle_rate(grid, chs, seconds_budget, steps, warmup, threads):
    """voxel-steps/s of the CPU oracle (oracle/: plain PyTorch fp32 restatement of the reference's mltools
    path): one reverse sampler step of one realisation per bench step.  When a 128^3 step does not fit the
    time budget the sample is a 64^3 box of the same network (conv cost is linear in voxels)."""
    from oracle.unet_ref import CUNet as RefNet
    from oracle.vdm_ref import VDM as RefVDM
    torch.set_num_threads(threads)

    def run(n, n_steps, n_warm):
        torch.manual_seed(42)
        net = RefNet(**model_kwargs(n, chs)).eval()
        vdm = RefVDM(net).eval()
        x, cond, params = synthetic_batch(1, n, 42)
        z = torch.randn_like(x)
        ts = torch.linspace(1.0, 0.0, 1001)
        times = []
        with torch.no_grad():
            for i in range(n_warm + n_steps):
                t0 = time.perf_counter()
                z = vdm.sample_zs_given_zt(zt=z, t=ts[i], s=ts[i + 1], s_conditioning=cond, v_conditionings=[params])
                if i >= n_warm:
                    times.append(time.perf_counter() - t0)
        return times

    probe = run(64, 1, 1)[0]
    est_full = probe * 8.0
    if est_full * (steps + warmup) <= seconds_budget:
        n, label = grid, f"{steps} reverse steps of 1 realisation at {grid}^3 (the full workload's per-step unit)"
        times = run(grid, steps, warmup)
    else:
        fit = max(1, int(seconds_budget / max(probe, 1e-3)) - warmup)
        k = max(1, min(steps, fit))
        n, label = 64, f"{k} reverse steps of 1 realisation on a 64^3 box of the same network (128^3 would exceed the time budget)"
        times = run(64, k, min(warmup, 1))
    sec = sum(times) / len(times)
    return (n ** 3) / sec, sec, label, len(times)


def parity_leg(net, vdm, dev, grid, chs):
    """Parity of the BENCHMARKED configuration, measured in the bench run: the oracle (oracle/unet_ref.py + vdm_ref.py,
    CPU fp32) gets the benchmarked network's weights and runs one denoiser call and one reverse step of one realisation
    at the full grid with injected noise; the CUDA path runs the same.  Reported as relative L2 (tolerance 1e-2: bf16
    activations, BASELINE.json north_star)."""
    from oracle.unet_ref import CUNet as RefNet
    from oracle.vdm_ref import VDM as RefVDM
    net.invalidate_packed()
    ref = RefNet(**model_kwargs(grid, chs)).eval()
    ref.load_state_dict({k: v.detach().cpu() for k, v in net.state_dict().items()}, strict=True)
    ref_vdm = RefVDM(ref).eval()
    g = torch.Generator().manual_seed(7)
    x, cond, params = synthetic_batch(1, grid, 4321)
    noise = torch.randn(x.shape, generator=g)
    t, s_ = torch.tensor(0.62), torch.tensor(0.616)
    with torch.no_grad():
        t_net = torch.tensor([0.37])
        want = ref(x, t=t_net, s_conditioning=cond, v_conditionings=[params])
        got = net(x.to(dev), t=t_net.to(dev), s_conditioning=cond.to(dev), v_conditionings=[params.to(dev)]).cpu()
        zs_r = ref_vdm.sample_zs_given_zt(zt=x, t=t, s=s_, noise=noise, s_conditioning=cond, v_conditionings=[params])
        zs = vdm.sample_zs_given_zt(zt=x.to(dev), t=t, s=s_, noise=noise.to(dev), s_conditioning=cond.to(dev),
                                    v_conditionings=[params.to(dev)]).cpu()
    rel = lambda a, b: ((a - b).norm() / b.norm()).item()
    return {"denoiser_rel_l2": rel(got, want), "step_rel_l2": rel(zs, zs_r), "tolerance": 1e-2,
            "against": f"oracle/ (CPU fp32) with the benchmarked weights, 1 realisation at {grid}^3 chs={chs}"}


def torch_gpu_leg(args, dev, ours_ms_per_step, ours_train_ms):
    """Stock PyTorch on the SAME B200 (SURVEY.md section 2.3: the bar a user of the reference would compare with): the
    oracle's modules on cuda, i.e. cuDNN conv3d + ATen GroupNorm/SiLU, eager launches, cudnn.benchmark on, in three
    settings -- "tf32" (fp32 tensors, TF32 convs: what the reference's scripts run, torch.set_float32_matmul_precision
    ("medium"), trainVDM3D128_...:18), "bf16" (torch.autocast) and "bf16_cl3d" (autocast + channels_last_3d).  Same work as
    our arms: one reverse step of `batch` realisations, and one VDM training step (loss fwd + bwd + clip 0.5 + AdamW) of
    `train_batch` samples; CUDA events.  The ratios are taken against the FASTEST stock setting.  None of this
    repository's kernels run here."""
    from oracle.unet_ref import CUNet as RefNet
    from oracle.vdm_ref import LightVDM as RefLight
    from oracle.vdm_ref import VDM as RefVDM
    grid, chs = args.grid, args.chs
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.benchmark = True
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cuda.matmul.allow_tf32 = True
    out = {"what": "oracle modules on cuda:0 (stock PyTorch: cuDNN conv3d + ATen GroupNorm/SiLU), eager launches, "
                   "cudnn.benchmark; settings tf32 (the reference's own), bf16 autocast, bf16 autocast + channels_last_3d",
           "torch": torch.__version__, "cudnn": torch.backends.cudnn.version(), "sampling": {}, "training": {}}
    settings = {"tf32": (False, torch.contiguous_format), "bf16": (True, torch.contiguous_format),
                "bf16_cl3d": (True, torch.channels_last_3d)}

    def timed(fn, warm, iters):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / iters

    for name, (autocast, fmt) in settings.items():
        try:
            torch.manual_seed(42)
            net = RefNet(**model_kwargs(grid, chs)).to(dev).to(memory_format=fmt).eval()
            vdm = RefVDM(net).to(dev).eval()
            x, cond, params = synthetic_batch(args.batch, grid, 42, device=dev)
            cond = cond.contiguous(memory_format=fmt)
            state = {"z": torch.randn_like(x)}
            ts = torch.linspace(1.0, 0.0, 1001, device=dev)
            it = [0]

            def sample_step():
                i = it[0] % 1000
                it[0] += 1
                with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    state["z"] = vdm.sample_zs_given_zt(zt=state["z"], t=ts[i], s=ts[i + 1], s_conditioning=cond,
                                                        v_conditionings=[params]).float()

            ms = timed(sample_step, 3, 5)
            out["sampling"][name] = {"ms_per_step": ms, "value": args.batch * grid ** 3 / (ms * 1e-3), "unit": UNIT,
                                     "realisations": args.batch}
            del vdm, net, state
            torch.cuda.empty_cache()
            if ours_train_ms is not None:
                torch.manual_seed(42)
                net = RefNet(**model_kwargs(grid, chs)).to(dev).to(memory_format=fmt).train()
                light = RefLight(net).to(dev).train()
                opt = torch.optim.AdamW(light.parameters(), lr=3.0e-4, fused=True)
                xb, cb, pb = synthetic_batch(args.train_batch, grid, 4242, device=dev)
                batch = {"x": xb, "conditioning": cb.contiguous(memory_format=fmt), "conditioning_values": [pb]}

                def train_step():
                    opt.zero_grad(set_to_none=True)
                    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                        loss, _ = light.get_loss(batch)
                    loss.backward()
                    torch.nn.utils.clip_grad_norm_(light.parameters(), 0.5)
                    opt.step()

                ms_t = timed(train_step, 3, 5)
                out["training"][name] = {"ms_per_step": ms_t, "value": args.train_batch / (ms_t * 1e-3), "unit": "samples/s",
                                         "batch": args.train_batch}
                del light, net, opt, batch
        except Exception as exc:                         # e.g. cuDNN has no engine for a layer in this setting
            out.setdefault("errors", {})[name] = f"{type(exc).__name__}: {exc}"[:300]
        torch.cuda.empty_cache()
    torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    if out["sampling"]:
        best = min(out["sampling"], key=lambda k: out["sampling"][k]["ms_per_step"])
        out["fastest_sampling_setting"] = best
        out["vs_torch_gpu_sampling"] = out["sampling"][best]["ms_per_step"] / ours_ms_per_step
    if out["training"]:
        best = min(out["training"], key=lambda k: out["training"][k]["ms_per_step"])
        out["fastest_training_setting"] = best
        out["vs_torch_gpu_training"] = out["training"][best]["ms_per_step"] / ours_train_ms
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    value, sec, label, k = cpu_oracle_rate(args.grid, args.chs, 240.0, args.steps, args.warmup, threads)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": k,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"VDM 3D c_c {args.grid}^3 chs={args.chs} reverse ancestral sampling, CPU oracle port",
                       "sample": label},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": label},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ---------------------------------------------------------------------------------------------------------
def run_b200(args, rank, world, local_rank):
    import torch.distributed as dist

    from vdm4cdm_b200 import _C, ops
    from vdm4cdm_b200.networks import CUNet
    from vdm4cdm_b200.vdm_model import LightVDM

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    _C.check(_C.lib().vdm_device_supported(local_rank), "vdm_device_supported")   # fails loudly off-B200
    grid, chs, batch = args.grid, args.chs, args.batch
    voxels = grid ** 3
    torch.manual_seed(42)
    net = CUNet(**model_kwargs(grid, chs))
    model = LightVDM(score_model=net, draw_figure=None, gamma_max=13.3, learning_rate=3.0e-4).to(dev).eval()
    vdm = model.model
    x, cond, params = synthetic_batch(batch, grid, 42 + rank)
    rids = [rank * batch + i for i in range(batch)]

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- device-resident throughput: K graph-replayed steps of a 1000-step chain ----
    n_chain = max(1000, args.warmup + args.steps + 2)
    sess = vdm.session(batch, n_chain, dev, seed=42, realisation_ids=rids, s_conditioning=cond.to(dev),
                       v_conditionings=[params.to(dev)])
    for _ in range(max(args.warmup, 3)):          # includes the eager step and the graph capture
        sess.step()
    clocks = ClockSampler(local_rank)
    barrier()
    clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        sess.step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clock_info = clocks.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = t.item()
    value = world * batch * voxels * args.steps / (ms_max * 1e-3)
    launches = sess.kernels_per_step * args.steps
    assert torch.isfinite(sess.z).all(), "sampler state went non-finite"
    if args.dump_outputs and rank == 0:
        # the latent after the last timed step (what the chain hands on) and the denoiser output that step used
        dump_outputs(args.dump_outputs, {"z": sess.z, "eps": sess.eps})

    # ---- end to end through the public API: host conditioning in, host sample out ----
    # one public-API call = one whole chain: the reference's default length (LightVDM.draw_samples(n_sampling_steps=250),
    # model_test.ipynb:667); conditioning goes in and the samples come out once per chain
    n_e2e = max(args.steps, args.e2e_chain)
    cond_h, params_h = cond.pin_memory(), params.pin_memory()
    out_h = torch.empty((batch, 1, grid, grid, grid), dtype=torch.float32).pin_memory()

    def user_call():
        c = cond_h.to(dev, non_blocking=True)
        p = params_h.to(dev, non_blocking=True)
        xs = model.draw_samples(batch_size=batch, n_sampling_steps=n_e2e, s_conditioning=c, v_conditionings=[p],
                                seed=42, realisation_ids=rids)
        out_h.copy_(xs, non_blocking=True)
        torch.cuda.synchronize(dev)

    user_call()                                     # first call builds the session and its graph
    barrier()
    t0 = time.perf_counter()
    user_call()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * batch * voxels * n_e2e / t.item()
    h2d = (cond_h.numel() * 4 + params_h.numel() * 4) / n_e2e
    d2h = out_h.numel() * 4 / n_e2e

    # ---- BASELINE.json configs[4] scaled down: ensemble sampling -> calc_SS statistics gathered on rank 0 ----
    pipeline = pipeline_leg(args, model, dev, rank, world, x, cond, params, rids)
    if rank != 0:
        if not args.no_train:
            train_leg(args, model, net, dev, rank, world, 1.0)
        return
    # ---- roofline of the dominant kernels (conv3d_planar_kernel, conv3d_march_kernel): CUDA events around every conv launch ----
    peaks, peak_kind = measured_peaks()
    vdm.use_cuda_graph = False
    sess2 = vdm.session(batch, n_chain, dev, seed=42, realisation_ids=rids, s_conditioning=cond.to(dev),
                        v_conditionings=[params.to(dev)])
    sess2.step()
    prof_steps = 3
    step_records, step_ms = [], []
    for _ in range(prof_steps):
        records = []
        ops.set_conv_profiler(records)
        torch.cuda.synchronize(dev)
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s0.record()
        sess2.step()
        s1.record()
        torch.cuda.synchronize(dev)
        ops.set_conv_profiler(None)
        step_records.append(records)
        step_ms.append(s0.elapsed_time(s1))
    # the fastest of the profiled steps (event-bracketed eager launches pick up host hiccups: one slow launch
    # tripled a layer's time in r01v)
    sums = [sum(r[0].elapsed_time(r[1]) for r in recs) for recs in step_records]
    best = min(range(prof_steps), key=lambda i: sums[i])
    records = step_records[best]
    conv_ms = sums[best]
    per_layer = {}
    for r in records:
        e = per_layer.setdefault(r[3], [0.0, 0.0, 0])
        e[0] += r[0].elapsed_time(r[1])
        e[1] += r[2]
        e[2] += 1
    for k, (ms_l, fl, n) in sorted(per_layer.items(), key=lambda kv: -kv[1][0]):
        print(f"[conv] {k:42s} x{n}: {ms_l:7.3f} ms/step {fl / (ms_l * 1e-3) / 1e12:7.1f} TFLOP/s", file=sys.stderr)
    vdm.use_cuda_graph = True
    eager_step_ms = step_ms[best]
    conv_flops = net.conv_flops_per_sample() * batch
    achieved = conv_flops / (conv_ms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        # DRAM read + write of one step's conv launches (ncu --set full), valid for the workload it was captured on
        # (a capture of another grid / batch / set of conv launches does not apply: traffic stays null)
        if tj.get("grid", 128) == args.grid and tj.get("realisations_per_gpu") == args.batch and \
                tj.get("conv_launches_per_step") == len(records):
            traffic = tj.get("conv_dram_bytes_per_step")
    roofline = {"kernel": "conv3d_planar_kernel + conv3d_march_kernel (all conv launches of one step)", "bound": "tensor",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_kind})", "traffic": traffic,
                "traffic_source": "profiles/roofline_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum of the conv "
                                  "launches of one step of this workload; not measurable inside the timed run)" if traffic else None,
                "algorithmic_flops_per_step": conv_flops, "conv_launches_per_step": len(records),
                "conv_ms_per_step": conv_ms, "conv_share_of_eager_step": conv_ms / eager_step_ms}

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample; parity of this very network ----
    cpu, parity = None, None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, sec, label, k = cpu_oracle_rate(grid, chs, 30.0, 2, 1, threads)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "sample": label, "s_per_step": sec}
        model.eval()
        parity = parity_leg(net, vdm, dev, grid, chs)

    # ---- training step (BASELINE.json configs[1]: trainVDM3D128..._lowbatch, batch_size=2 per GPU) ----
    train = None
    if not args.no_train:
        train = train_leg(args, model, net, dev, rank, world, peak)

    # ---- P(k) / r(k) of generated fields (SURVEY.md section 8d metric iii) ----
    pk = pk_leg(grid, dev, peaks)

    # ---- other BASELINE.json configurations (configs[2], configs[3]): one training step each, 1 GPU ----
    other = None
    if world == 1 and not args.no_train and not args.no_other_configs:
        other = other_configs_leg(dev)

    # ---- stock PyTorch (cuDNN / ATen) on the same GPU: the oracle's modules under bf16 autocast ----
    torch_gpu = None
    if world == 1 and not args.no_torch_gpu_baseline:
        torch_gpu = torch_gpu_leg(args, dev, ms_max / args.steps, None if train is None else train["ms_per_step"])

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"VDM 3D c_c {grid}^3 chs={chs} (configs.yaml VDM_*_c_c_128), reverse ancestral "
                                   f"sampling, {batch} realisations per GPU, step of a 1000-step chain",
                       "grid": grid, "realisations_per_gpu": batch, "parallelism": f"{world} independent shards of realisations",
                       "l2": "no flush: one step streams >3 GB of activations per realisation, far above the 126 MB L2",
                       "cuda_graph": True},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "call": f"LightVDM.draw_samples(batch_size={batch}, n_sampling_steps={n_e2e}) with pinned host "
                            "conditioning in and the sample copied back to pinned host memory"},
            "gpu_launches": launches, "clocks": clock_info, "roofline": roofline,
            "conv_tflops": achieved}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if parity is not None:
        line["parity"] = parity
    if train is not None:
        line["train"] = train
        for k in ("replicas_identical", "grad_vs_1gpu_rel"):       # N > 1: correctness of the data-parallel step on hardware
            if k in train:
                line[k] = train[k]
    line["pk"] = pk
    if pipeline is not None:
        line["pipeline"] = pipeline
    if other is not None:
        line["other_configs"] = other
    if torch_gpu is not None:
        line["torch_gpu_baseline"] = torch_gpu
        for k in ("vs_torch_gpu_sampling", "vs_torch_gpu_training"):
            if k in torch_gpu:
                line[k] = torch_gpu[k]
    emit(line)


def pipeline_leg(args, model, dev, rank, world, x, cond, params, rids):
    """BASELINE.json configs[4], scaled down to a bench-sized chain: every rank draws its `batch` realisations with
    ``draw_samples`` (``--pipeline-steps`` reverse steps instead of 1000), computes calc_SS.py's P(k) of each sample and
    r(k) against its truth field on the GPU, and rank 0 gathers the (kmax,) vectors of all world x batch realisations.
    Wall time over the whole pipeline, max over ranks."""
    import torch.distributed as dist

    from vdm4cdm_b200 import utils
    from vdm4cdm_b200.dataset import ALPHAS_3D, NORMALIZATIONS_3D, unnorm_func
    n = args.pipeline_steps
    if n <= 0:
        return None
    mu, sd = NORMALIZATIONS_3D["Mcdm"]
    un = lambda f: unnorm_func(f, ALPHAS_3D["Mcdm"], mu, sd)
    c, pv, truth = cond.to(dev), params.to(dev), x.to(dev)

    def run():
        xs = model.draw_samples(batch_size=args.batch, n_sampling_steps=n, s_conditioning=c, v_conditionings=[pv], seed=43,
                                realisation_ids=rids)
        # random-init weights amplify z by alpha_0/alpha_1 ~ 770 over a chain: clip to the range of the normalised data
        # (the +-4 of draw_figure's histograms, src/utils.py:161) so that 10**x stays finite; the work is unchanged
        s_un, t_un = un(xs.clamp(-4.0, 4.0)), un(truth)
        s_un = (s_un / s_un.sum((2, 3, 4), keepdim=True)).contiguous()          # calc_SS.py:67-70
        t_un = (t_un / t_un.sum((2, 3, 4), keepdim=True)).contiguous()
        _, pk_s, _ = utils.pk(s_un)
        _, cc = utils.get_ccs(s_un, t_un)
        stats = torch.stack([pk_s.float(), cc.float()], dim=1)                     # (batch, 2, kmax)
        if world > 1:
            out = [torch.empty_like(stats) for _ in range(world)] if rank == 0 else None
            dist.gather(stats, out, dst=0)
            stats = torch.cat(out) if rank == 0 else stats
        return stats

    run()                                               # builds the session / graph for this chain length
    torch.cuda.synchronize(dev)
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    stats = run()
    torch.cuda.synchronize(dev)
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    return {"what": f"{world * args.batch} realisations x {n} reverse steps at {args.grid}^3 -> P(k) and r(k) vs truth per "
                    "realisation (calc_SS.py) -> gathered on rank 0",
            "realisations": world * args.batch, "steps": n, "wall_s": t.item(), "gathered_shape": list(stats.shape),
            "finite": bool(torch.isfinite(stats).all()), "voxel_steps_per_s": world * args.batch * args.grid ** 3 * n / t.item()}


def other_configs_leg(dev):
    """One graph-replayed training step of BASELINE.json configs[2] (SFM 3D c_c at 160^3, chs [32,64,128,256], batch 4:
    trainSFM3D160_...:60,68) and configs[3] (VDM 3D c_c at 224^3, chs [16,32,64,128], batch 2: trainVDM3D224_...:60,72):
    samples/s, conv TFLOP/s against the sustained bf16 peak, peak memory.  Synthetic Gaussian fields."""
    from vdm4cdm_b200.networks import CUNet
    from vdm4cdm_b200.sfm_model import LightSFM
    from vdm4cdm_b200.trainer import Trainer
    from vdm4cdm_b200.vdm_model import LightVDM
    peaks, _ = measured_peaks()
    peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops")))
    out = {}
    for key, kind, n, chs, batch in (("sfm160", "SFM", 160, [32, 64, 128, 256], 4), ("vdm224", "VDM", 224, [16, 32, 64, 128], 2)):
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
        torch.manual_seed(42)
        net = CUNet(**model_kwargs(n, chs))
        model = (LightVDM(score_model=net, gamma_max=13.3) if kind == "VDM" else LightSFM(velocity_model=net)).to(dev)
        trainer = Trainer(model, gradient_clip_val=0.5)
        x, cond, params = synthetic_batch(batch, n, 42, device=dev)
        b = {"x": x, "conditioning": cond, "conditioning_values": [params]} if kind == "VDM" else \
            {"x0": cond, "x1": x, "conditioning_values": [params]}
        losses = [trainer.training_step(b).item() for _ in range(5)]            # 3 eager + capture + replay
        steps = 8
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(steps):
            loss = trainer.training_step(b)
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / steps
        flops = 3.0 * net.conv_flops_per_sample() * batch        # fwd + dgrad + wgrad (conv_in's dgrad included: z needs it)
        out[key] = {"config": f"{kind} 3D c_c {n}^3 chs={chs} batch {batch}", "ms_per_step": ms, "samples_per_s": batch / (ms * 1e-3),
                    "steps": steps, "peak_mem_gib": torch.cuda.max_memory_allocated(dev) / 2 ** 30,
                    "step_tflops_conv_algorithmic": flops / (ms * 1e-3) / 1e12,
                    "step_frac_of_peak": flops / (ms * 1e-3) / 1e12 / peak,
                    "first_loss": losses[0], "last_loss": loss.item(), "cuda_graph": trainer._graph is not None}
        del trainer, model, net, b, x, cond, params
    torch.cuda.empty_cache()
    return out


def ddp_check(model, trainer, batch, dev, rank, world):
    """Correctness of the data-parallel training step ON THE HARDWARE (N > 1), after the timed steps:
      * ``replicas_identical``: an exact integer checksum of every rank's flat parameter bucket (fp32 bit patterns summed
        in int64) and of its AdamW moments is all-gathered and must be equal on all ranks;
      * ``grad_vs_1gpu_rel``: every rank back-propagates ITS micro-batch (fixed times / noise, dropout off) and the flat
        gradient bucket is all-reduced and averaged exactly as the step does; rank 0 then recomputes the same global
        batch alone, micro-batch by micro-batch, accumulating into the same bucket.  Relative L2 of the difference (only
        the summation order of fp32 atomics / the NCCL reduction tree differs)."""
    import torch.distributed as dist

    def checksum(t):
        return t.view(torch.int32).to(torch.int64).sum()

    mine = torch.stack([checksum(trainer.buckets.flat_param), checksum(trainer.exp_avg), checksum(trainer.exp_avg_sq)])
    allc = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(allc, mine)
    identical = all(torch.equal(c, allc[0]) for c in allc)

    flat = {"x": batch["x"], "conditioning": batch["conditioning"], "conditioning_values": batch["conditioning_values"][0]}
    gathered = {}
    for k, v in flat.items():
        parts = [torch.empty_like(v) for _ in range(world)]
        dist.all_gather(parts, v.contiguous())
        gathered[k] = parts
    g = torch.Generator(device=dev)
    bsz = batch["x"].shape[0]

    def micro_grad(r):
        g.manual_seed(1000 + r)
        xb = gathered["x"][r]
        noise = torch.randn(xb.shape, generator=g, device=dev)
        noise0 = torch.randn(xb.shape, generator=g, device=dev)
        times = torch.remainder(torch.rand((), generator=g, device=dev) + torch.arange(bsz, device=dev) / bsz, 1.0)
        b = {"x": xb, "conditioning": gathered["conditioning"][r], "conditioning_values": [gathered["conditioning_values"][r]]}
        loss, _ = model.get_loss(b, noise=noise, noise0=noise0, times=times)
        loss.backward()                                   # accumulates into the flat gradient bucket

    model.eval()                                          # dropout off; gradients still flow (grad mode is on)
    trainer.buckets.zero_grad()
    micro_grad(rank)
    dist.all_reduce(trainer.buckets.flat_grad, op=dist.ReduceOp.SUM)
    g_multi = trainer.buckets.flat_grad.clone() / world
    rel = torch.zeros(1, dtype=torch.float64, device=dev)
    if rank == 0:
        trainer.buckets.zero_grad()
        for r in range(world):
            micro_grad(r)
        g_single = trainer.buckets.flat_grad / world
        rel[0] = ((g_multi - g_single).double().norm() / g_single.double().norm()).item()
    dist.broadcast(rel, src=0)
    trainer.buckets.zero_grad()
    model.train()
    return {"replicas_identical": bool(identical), "grad_vs_1gpu_rel": rel.item()}


def pk_leg(grid, dev, peaks):
    """fields/s of utils.pk (cuFFT R2C + k-shell binning) and utils.get_ccs on 16 mass-like 128^3 fields; the binning
    pass is HBM-bound: algorithmic bytes = 4 N^3 (field read by the FFT) + 16 N^2 (N/2+1) (spectrum written and read)."""
    from vdm4cdm_b200 import utils
    n_fields = 16
    g = torch.Generator(device=dev).manual_seed(7)
    x = torch.randn((n_fields, 1, grid, grid, grid), generator=g, device=dev)
    mass = 10.0 ** (x * 0.552 + 10.019) - 1.0                         # calc_SS.py:67-70 input definition
    mass = mass / mass.sum((2, 3, 4), keepdim=True)
    other = 0.7 * mass + 0.3 * mass.flip(2)

    def timed(fn, iters=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / iters

    ms_pk = timed(lambda: utils.pk(mass))
    ms_cc = timed(lambda: utils.get_ccs(mass, other))
    bytes_field = 4.0 * grid ** 3 + 16.0 * grid * grid * (grid // 2 + 1)
    hbm = float(peaks.get("hbm_gbs", 6550.0))
    gbs = n_fields * bytes_field / (ms_pk * 1e-3) / 1e9
    return {"metric": f"P(k) fields/s at {grid}^3 (cuFFT R2C + binning, {n_fields} fields per call)",
            "value": n_fields / (ms_pk * 1e-3), "unit": "fields/s", "ms_per_call": ms_pk,
            "get_ccs_pairs_per_s": n_fields / (ms_cc * 1e-3),
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm, "unit": "GB/s", "frac": gbs / hbm,
                         "algorithmic_bytes_per_field": bytes_field}}


def train_leg(args, model, net, dev, rank, world, peak_tflops):
    """train samples/s: LightVDM.training_step (VDM loss fwd + bwd) + gradient all-reduce + clip + AdamW on
    `args.train_batch` samples per GPU; device-resident (CUDA events, max over ranks) and end to end (pinned
    host batch in, loss scalar out, every step)."""
    import torch.distributed as dist

    from vdm4cdm_b200 import ops
    from vdm4cdm_b200.trainer import Trainer

    grid, batch = args.grid, args.train_batch
    model.model.__dict__.get("_sessions", {}).clear()          # release the sampler's buffers
    net._arena.bufs.clear()
    torch.cuda.empty_cache()
    model.train()
    trainer = Trainer(model, gradient_clip_val=0.5)
    x, cond, params = synthetic_batch(batch, grid, 4242 + rank)
    host = {"x": x.pin_memory(), "conditioning": cond.pin_memory(), "conditioning_values": params.pin_memory()}

    def to_dev():
        return {"x": host["x"].to(dev, non_blocking=True), "conditioning": host["conditioning"].to(dev, non_blocking=True),
                "conditioning_values": [host["conditioning_values"].to(dev, non_blocking=True)]}

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    resident = to_dev()
    staging = to_dev()                           # device staging buffers of the end-to-end loop (allocated once)

    def h2d():
        staging["x"].copy_(host["x"], non_blocking=True)
        staging["conditioning"].copy_(host["conditioning"], non_blocking=True)
        staging["conditioning_values"][0].copy_(host["conditioning_values"], non_blocking=True)
        return staging

    n_steps, n_warm = args.train_steps, 3
    losses = []
    for _ in range(n_warm):
        losses.append(trainer.training_step(resident))
    for _ in range(2):                          # the step after the warm-up captures the CUDA graph; one replay
        losses.append(trainer.training_step(resident))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_steps):
        losses.append(trainer.training_step(resident))
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = t.item() / n_steps
    loss_vals = [float(l) for l in losses]
    assert all(v == v and abs(v) < 1e9 for v in loss_vals), f"training loss went non-finite: {loss_vals}"
    # end to end: pinned host batch -> device, step, loss scalar back, every step
    barrier()
    t0 = time.perf_counter()
    marks = []
    for _ in range(n_steps):
        ta = time.perf_counter()
        dev_batch = h2d()
        tb = time.perf_counter()
        loss = trainer.training_step(dev_batch)
        tc = time.perf_counter()
        loss_host = loss.item()
        marks.append((tb - ta, tc - tb, time.perf_counter() - tc))
    e2e_s = time.perf_counter() - t0
    if rank == 0:
        print("[train e2e] per step (h2d issue, step issue, wait for loss) ms: " +
              "; ".join("%.1f %.1f %.1f" % (a * 1e3, b * 1e3, c * 1e3) for a, b, c in marks), file=sys.stderr)
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t.item() * 1e3 / n_steps
    # conv kernels of one training step, by kind (CUDA events around each launch).  Every rank runs the step (it
    # contains the gradient all-reduce); only rank 0 keeps the records.
    records = []
    ops.set_conv_profiler(records if rank == 0 else None)
    n0 = ops.launch_count()
    trainer._eager_step(resident)               # same kernels as the captured step, launched one by one
    launches = ops.launch_count() - n0
    torch.cuda.synchronize(dev)
    ops.set_conv_profiler(None)
    check = ddp_check(model, trainer, resident, dev, rank, world) if world > 1 else {}
    if rank != 0:
        return None
    kinds = {"fprop": [0.0, 0.0], "dgrad": [0.0, 0.0], "wgrad": [0.0, 0.0]}
    per_layer = {}
    for r in records:
        kind = "wgrad" if r[3].startswith("wgrad") else ("dgrad" if r[3].startswith("dgrad") else "fprop")
        ms_r = r[0].elapsed_time(r[1])
        kinds[kind][0] += ms_r
        kinds[kind][1] += r[2]
        e = per_layer.setdefault(r[3], [0.0, 0.0, 0])
        e[0] += ms_r; e[1] += r[2]; e[2] += 1
    for k, (ms_l, fl, n) in sorted(per_layer.items(), key=lambda kv: -kv[1][0])[:24]:
        print(f"[train conv] {k:48s} x{n}: {ms_l:7.3f} ms/step {fl / (ms_l * 1e-3) / 1e12:7.1f} TFLOP/s", file=sys.stderr)
    conv_ms = sum(v[0] for v in kinds.values())
    conv_fl = sum(v[1] for v in kinds.values())
    return {"metric": "train samples/s (VDM 3D c_c 128^3, fwd+bwd+allreduce+clip+AdamW)",
            "value": world * batch / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "steps": n_steps, "warmup": n_warm,
            "global_batch": world * batch, "batch_per_gpu": batch, "scaling": "weak",
            "e2e": {"value": world * batch / (e2e_ms * 1e-3), "unit": "samples/s",
                    "h2d_bytes_per_step": sum(v.numel() * 4 for v in host.values()), "d2h_bytes_per_step": 4,
                    "call": "Trainer.training_step(batch) with a pinned host batch in and loss.item() out"},
            "gpu_launches_per_step": launches, "cuda_graph": trainer._graph is not None, "first_loss": loss_vals[0], "last_loss": loss_host,
            "parameters": trainer.buckets.numel,
            "conv": {k: {"ms": v[0], "tflops": (v[1] / (v[0] * 1e-3) / 1e12) if v[0] > 0 else None} for k, v in kinds.items()},
            "conv_tflops": conv_fl / (conv_ms * 1e-3) / 1e12, "conv_frac_of_peak": conv_fl / (conv_ms * 1e-3) / 1e12 / peak_tflops,
            "conv_share_of_step": conv_ms / ms, **check}


_REAL_STDOUT = None


def quiet_stdout():
    """stdout carries exactly ONE JSON line: everything libraries print there (NCCL prints its version banner on
    stdout) is routed to stderr at the file-descriptor level; ``emit`` writes to the saved descriptor."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8,
                    help="realisations sampled together per GPU (BASELINE.json configs[4]: 64 realisations over 8 GPUs)")
    ap.add_argument("--grid", type=int, default=128)
    ap.add_argument("--chs", type=int, nargs="+", default=[32, 64, 128, 256])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-chain", type=int, default=250, help="reverse steps of the end-to-end draw_samples call")
    ap.add_argument("--no-train", action="store_true", help="skip the training-step leg")
    ap.add_argument("--train-batch", type=int, default=2, help="training samples per GPU (reference: batch_size = 2)")
    ap.add_argument("--train-steps", type=int, default=20)
    ap.add_argument("--no-torch-gpu-baseline", action="store_true", help="skip the stock-PyTorch-on-GPU arm")
    ap.add_argument("--no-other-configs", action="store_true", help="skip the SFM 160^3 / VDM 224^3 training steps")
    ap.add_argument("--pipeline-steps", type=int, default=20, help="reverse steps of the scaled-down ensemble pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's latent z and denoiser output eps of the last timed step "
                         "as DIR/z.npy and DIR/eps.npy (float32; arrays above 2^22 elements as a fixed seeded sample)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl b200)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank),
                                timeout=datetime.timedelta(seconds=180))   # a desynchronised collective must fail fast
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
