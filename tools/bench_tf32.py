"""bf16 vs TF32 sampling steps of the VDM 3-D denoiser, and the reference modules under cuDNN TF32 on the same card.

    python tools/bench_tf32.py [--steps 20] [--out profiles/<name>.json]

For each workload (128^3 x 8 and 64^3 x 2, chs = (32, 64, 128, 256)) the two precisions of one CUNet run alternately,
a sampling step each time as a CUDA-graph replay of the SamplerSession, `--rounds` rounds of `--steps` timed steps per
precision (CUDA events around the steps).  The oracle (oracle/unet_ref.py, plain fp32 PyTorch modules with the same
weights) runs the denoiser eagerly on the GPU with torch.backends.cudnn.allow_tf32 = True: the reference's own precision
on the same card.  Conv TFLOP/s = algorithmic conv FLOPs of one forward (CUNet.conv_flops_per_sample) x batch / step time,
against the data sheet's 1,125 dense TF32 TFLOP/s (2,250 bf16) for one B200 at 1,000 W.  The card's name and power limit
are read in the same run.  Needs a GPU; there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK = {"bf16": 2250.0, "tf32": 1125.0}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def time_steps(sess, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        sess.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tf32.py needs a CUDA device")
    from oracle.unet_ref import CUNet as RefNet
    from vdm4cdm_b200.networks import CUNet
    from vdm4cdm_b200.vdm_model import VDM
    dev = torch.device("cuda:0")
    chs = (32, 64, 128, 256)
    result = {"card": card(), "chs": list(chs), "workloads": []}
    for grid, batch in ((128, 8), (64, 2)):
        torch.manual_seed(0)
        kw = dict(shape=(1, grid, grid, grid), chs=chs, s_conditioning_channels=0, v_conditioning_dims=[], t_conditioning=True)
        net = CUNet(**kw).to(dev).eval()
        vdm = VDM(net).to(dev).eval()
        flops = net.conv_flops_per_sample() * batch
        n_chain = 2 + args.rounds * args.steps + 1
        sessions = {}
        for prec in ("bf16", "tf32"):
            net.precision = prec
            sessions[prec] = vdm.session(batch, n_chain, dev, seed=1)
            vdm.__dict__.pop("_sessions", None)         # keep both sessions (the cache holds one)
            sessions[prec].step()                      # eager warm-up, then the graph capture
            sessions[prec].step()
        times = {"bf16": [], "tf32": []}
        for _ in range(args.rounds):
            for prec in ("bf16", "tf32"):
                net.precision = prec
                times[prec].append(time_steps(sessions[prec], args.steps))
        del sessions
        torch.cuda.empty_cache()
        w = {"grid": grid, "batch": batch, "conv_gflop_per_step": flops / 1e9}
        for prec in ("bf16", "tf32"):
            ms = min(times[prec])
            w[prec] = {"ms_per_step": ms, "ms_per_step_rounds": times[prec],
                       "conv_tflops": flops / ms / 1e9, "share_of_datasheet_peak": flops / ms / 1e9 / PEAK[prec]}
        # the oracle's modules on the GPU, eager, cuDNN TF32 (the reference scripts' default precision)
        ref = RefNet(**kw).to(dev).eval()
        ref.load_state_dict(net.state_dict(), strict=False)
        old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = True
        try:
            x = torch.randn((batch, 1, grid, grid, grid), device=dev)
            t = torch.rand(batch, device=dev)
            with torch.no_grad():
                for _ in range(2):
                    ref(x, t=t)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n = max(3, args.steps // 4)
                e0.record()
                for _ in range(n):
                    ref(x, t=t)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n
        finally:
            torch.backends.cudnn.allow_tf32 = old[0]
        w["oracle_cudnn_tf32_eager"] = {"ms_per_forward": ms, "conv_tflops": flops / ms / 1e9,
                                         "share_of_datasheet_peak": flops / ms / 1e9 / PEAK["tf32"]}
        del ref, net, vdm
        torch.cuda.empty_cache()
        result["workloads"].append(w)
        print(json.dumps(w), flush=True)
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
