#!/usr/bin/env python
"""Ensemble sampling with a trained (or random-init) 3-D conditional VDM: the reference's ``generate_3D.py``
(same positional CLI: model_name save_path runtype; its loop is generate_3D.py:43-97) on the B200-native path.

Differences, all in how the work is scheduled, not in what is computed:
  * realisations are independent units: realisation r of a test field goes to rank r mod world_size
    (``torchrun --nproc-per-node N scripts/generate_3D.py ...``), several per GPU at a time (``--batch``), and its
    noise stream is keyed by (seed, r) -- the saved ensemble does not depend on N or on the batch size;
  * the reverse loop replays one captured CUDA graph per step (vdm4cdm_b200.vdm_model.SamplerSession);
  * ``--synthetic`` stands in for the CAMELS CV test set (see scripts/_common.py).
Output: ``save_path/gen_{count}.npy`` with shape (rep, 1, N, N, N), as the reference writes it
(``{name}_{rep}.npy`` for the 1P run types of ``generate_3D_1P.py``, which is this file's ``main("1P")``).
"""
import argparse
import os

import numpy as np
import yaml

from _common import ROOT, init_distributed, synthetic_batch

import torch
import torch.distributed as dist

from vdm4cdm_b200 import utils
from vdm4cdm_b200.trainer import shard_indices


# generate_3D_1P.py:44-45: the five members of the CAMELS 1P set the reference samples (fiducial, Omega_m -2/+2,
# A_SN1 -3/+3), by index into the 1P test loader, and the names its output files carry
ONE_P_INDICES = [0, 4, 7, 23, 28]
ONE_P_NAMES = ["fid", "Om_m2", "Om_p2", "ASN1_m3", "ASN1_p3"]


def main(mode="CV"):
    ap = argparse.ArgumentParser(description="Generate 3D CDM")
    ap.add_argument("model_name", type=str, help="Model name (an entry of configs.yaml)")
    ap.add_argument("save_path", type=str, help="Save path")
    ap.add_argument("runtype", type=str, help="CV_12_12 (12 fields x 12 realisations) or CV_1_128 (1 field x 128); "
                    "generate_3D_1P.py: 1P_24 or 1P_128 (5 one-parameter-variation fields x 24 / 128)")
    ap.add_argument("--synthetic", action="store_true", help="synthetic conditioning fields instead of the CAMELS CV set")
    ap.add_argument("--data-root", default=os.environ.get("VDM4CDM_DATA_ROOT"),
                    help="directory with the CAMELS test grids and parameter files (vdm4cdm_b200.dataset.AstroDataModule)")
    ap.add_argument("--n-sampling-steps", type=int, default=250, help="reference default (model_test.ipynb:667)")
    ap.add_argument("--batch", type=int, default=2, help="realisations sampled together on one GPU")
    ap.add_argument("--rep", type=int, default=None, help="override the number of realisations per field")
    ap.add_argument("--fields", type=int, default=None, help="override the number of test fields")
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--allow-random-init", action="store_true",
                    help="smoke runs only: sample from random weights when the configured ckpt_path does not exist "
                         "(default: raise, like the reference's torch.load)")
    ap.add_argument("--configs", default=os.path.join(ROOT, "configs.yaml"))
    ap.add_argument("--precision", choices=["bf16", "tf32"], default="bf16",
                    help="denoiser precision: bf16 activations (default) or fp32 activations with TF32 convs, the "
                         "reference's cuDNN TF32 class of accuracy (A/B comparisons of the generated statistics)")
    args = ap.parse_args()
    if "SFM" in args.model_name:
        raise NotImplementedError("This model is not implemented yet")       # generate_3D.py:16-17
    assert args.runtype in (["CV_12_12", "CV_1_128"] if mode == "CV" else ["1P_24", "1P_128"])
    configs = yaml.safe_load(open(args.configs))
    assert args.model_name in configs, f"{args.model_name} is not in {args.configs}"
    config = configs[args.model_name]
    rank, world, device = init_distributed()
    if rank == 0:
        os.makedirs(args.save_path, exist_ok=True)
    model = utils.get_model(config, device=device, allow_random_init=args.allow_random_init).eval()
    if args.precision != "bf16":
        model.model.score_model.precision = args.precision        # the CUNet behind LightVDM -> VDM
    grid = int(config.get("cropsize", 128))
    n_params = int(config.get("conditioning_values", 6))
    if mode == "CV":
        n_fields, rep = (12, 12) if args.runtype == "CV_12_12" else (1, 128)
        field_ids = list(range(n_fields))
        names = [f"gen_{c}" for c in field_ids]                                   # generate_3D.py:66,94
    else:
        rep = 24 if args.runtype == "1P_24" else 128
        field_ids = ONE_P_INDICES
        names = [f"{n}_{rep}" for n in ONE_P_NAMES]                               # generate_3D_1P.py:70
    if args.fields:
        field_ids, names = field_ids[:args.fields], names[:args.fields]
    rep = args.rep or rep
    if args.rep and mode != "CV":
        names = [f"{n}_{args.rep}" for n in ONE_P_NAMES[:len(field_ids)]]
    if mode == "CV" and args.runtype == "CV_1_128" and not args.synthetic:
        field_ids = [2]                                                           # generate_3D.py:76 (sel=2)
    test_fields = {}
    if not args.synthetic:
        # generate_3D.py:43-47,71-75 / generate_3D_1P.py:52-53: test stage, batch 1, the CV or 1P set
        config.setdefault("data_params", {})
        config["data_params"].update(set_name="CV" if mode == "CV" else "1P", stage="test", batch_size=1)
        dm = utils.get_datamodule(config, data_root=args.data_root, device=device)
        for i_batch, batch in enumerate(dm.test_dataloader()):
            if i_batch in field_ids:
                test_fields[i_batch] = batch
            if i_batch >= max(field_ids):
                break
    for count, name in zip(field_ids, names):
        field = test_fields[count] if not args.synthetic else \
            synthetic_batch(1, grid, args.seed + 1000 + count, n_params)         # the same field on every rank
        if not n_params:
            field["conditioning_values"] = []                                     # generate_3D.py:56-57
        if rank == 0 and mode != "CV":
            print(name, "params", [v.tolist() for v in field["conditioning_values"]])
        mine = list(shard_indices(rep, rank, world))
        # One .npy per field, shape (rep, 1, N, N, N) as the reference writes it.  Every rank writes the rows of its own
        # realisations straight into the (memory-mapped) file: no dense ensemble buffer per rank and no collective over
        # it (r01 all-reduced a zero-filled (rep, 1, N^3) tensor from every rank: 1 GB at 128^3 x 128, 8.6 GB at 256^3).
        path = os.path.join(args.save_path, f"{name}.npy")
        if rank == 0:
            out = np.lib.format.open_memmap(path, mode="w+", dtype=np.float32, shape=(rep, 1, grid, grid, grid))
        if world > 1:
            dist.barrier()
        if rank != 0:
            out = np.lib.format.open_memmap(path, mode="r+")
        for i0 in range(0, len(mine), args.batch):
            ids = mine[i0:i0 + args.batch]
            b = len(ids)
            cond = field["conditioning"].to(device).expand(b, -1, -1, -1, -1).contiguous()
            vals = [v.to(device).expand(b, -1).contiguous() for v in field["conditioning_values"]]
            gen = model.draw_samples(batch_size=b, n_sampling_steps=args.n_sampling_steps, s_conditioning=cond,
                                     v_conditionings=vals, verbose=(rank == 0), seed=args.seed + count,
                                     realisation_ids=ids)
            out[ids] = gen.cpu().numpy()
        out.flush()
        del out
        if world > 1:
            dist.barrier()
        if rank == 0:
            print(f"{name}: saved {rep} realisations")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
