#!/usr/bin/env python
"""Kernel-development aid: time (or just run, for ncu) the MLP forward / weight-gradient kernels of one path over n voxels."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--path", default="piecewise", choices=["cuda_cores", "piecewise"])
    ap.add_argument("--n", type=int, default=256 ** 3)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    from diffus_b200 import ImpedanceEstimator, ops
    from diffus_b200.impedance import pack_params
    from diffus_b200.phantoms import mri_phantom
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)
    pk = pack_params(ImpedanceEstimator(1)).detach().to(dev)
    n = args.n
    x = (mri_phantom(256, "t2") / 1000.0).reshape(-1)[:n].contiguous().to(dev) if n <= 256 ** 3 else torch.rand(n, device=dev) * 3
    g = torch.randn(n, device=dev)
    path = {"cuda_cores": ops.MLP_PATH_CUDA_CORES, "piecewise": ops.MLP_PATH_PIECEWISE}[args.path]

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.iters
    ws = torch.empty((ops._lib.load().diffus_mlp_bwd_workspace_bytes(n),), dtype=torch.uint8, device=dev)
    gp = torch.zeros(1153, device=dev)
    with ops.mlp_path(path):
        f = timed(lambda: ops.mlp_fwd_impl(pk, x, None, 1e6, 400.0))
        b = timed(lambda: ops.mlp_bwd_impl(pk, x, None, g, 1e6, grad_params_out=gp, workspace=ws))
    print(json.dumps({"path": args.path, "n": n, "fwd_ms": f, "bwd_ms": b, "fwd_gb_per_s": n * 8 / f / 1e6, "bwd_gb_per_s": n * 8 / b / 1e6}))


if __name__ == "__main__":
    main()
