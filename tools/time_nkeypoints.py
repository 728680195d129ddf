"""Timings against the keypoint count (nkeypoints = 24, the tuned path, against 32 and 64): CUDA events with warm-up around
  - the detector forward at the bench shape (64 clips x 20 frames, G = 64, eval, no_grad), as frames/s;
  - the stage-1 training step (forward + backward + FusedAdam) at 24 clips x 10 frames, G = 64;
  - the 20-step HSVRNN roll-out (5 conditioned + 15 generated steps) at B = 1 and B = 24;
  - the stage-2 step (encode forward + backward + FusedAdam) at B = 24, T = 20.
The step-kernel column is derived from the launcher's routing rule (hsvrnn_step_impl in csrc/dynamics.cu), not observed.
Synthetic weights.

    python tools/time_nkeypoints.py [--ks 24,32,64] [--iters 5]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import neural_marionette_b200 as nm          # noqa: E402
from oracle import nm_oracle as O            # synthetic weights and clips only  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        pl = "unknown"
    return name, pl


def timed(fn, iters, warmup=2):
    for _ in range(warmup):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def build(K, G, train=False):
    hp = O.default_hparams(grid_size=G, nkeypoints=K)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(O.synthetic_state_dict(hp, seed=K))
    net = net.cuda().train(train)
    net.anneal(1)
    return net


def routed_step_kernel(K, B, S):
    """The HSVRNN step kernel hsvrnn_step_impl (csrc/dynamics.cu) routes to: a restatement of its rule, not a measurement."""
    if K <= 24 and S <= 10 and B <= 96:
        return "cluster"
    return "per-element"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ks", default="24,32,64")
    ap.add_argument("--iters", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    name, pl = card()
    print(f"GPU: {name}, power limit {pl}")
    G, clips, frames = 64, 64, 20
    raw = np.stack([O.synthetic_clip(1000 + b, frames, 20000) for b in range(clips)], 0)
    vox = nm.voxelize_raw_clips(raw, G)
    for K in [int(k) for k in args.ks.split(",")]:
        res = {"K": K}
        net = build(K, G)
        with torch.no_grad():
            ms = timed(lambda: net.kypt_detector(vox), args.iters)
        res["detector_frames_per_s"] = round(clips * frames / (ms / 1e3), 1)
        res["detector_ms"] = round(ms, 2)
        del net
        from neural_marionette_b200.optim import FusedAdam
        net = build(K, G, train=True)
        det = net.kypt_detector
        opt = FusedAdam([p for p in det.parameters() if p.requires_grad], lr=1e-4)
        v1 = vox[:24, :10].contiguous()

        def s1():
            opt.zero_grad(set_to_none=True)
            out = det(v1)
            (out["recon_loss"] + out["vol_fit_reg"]).backward()
            opt.step()
        res["stage1_step_ms"] = round(timed(s1, args.iters), 2)
        del net, opt
        net = build(K, 32)
        dm = net.dyna_module
        g = torch.Generator(device="cuda").manual_seed(K)
        with torch.no_grad():
            aff = net.kypt_detector.get_affinity()
        for B in (1, 24):
            kp = torch.rand(B, 5, K, 4, device="cuda", generator=g) * 1.2 - 0.6
            ec = torch.randn(5, 10, B, 128, device="cuda", generator=g)
            eg = torch.randn(15, B, 128, device="cuda", generator=g)
            with torch.no_grad():
                dm.encode(kp, aff)
                res[f"rollout_B{B}_ms"] = round(timed(lambda: dm.generate(kp, aff, Ttot=20, Tcond=5, eps_cond=ec,
                                                                          eps_gen=eg), args.iters * 2), 3)
            res[f"rollout_B{B}_kernel_by_rule"] = routed_step_kernel(K, B, 10)
        del net
        from neural_marionette_b200.optim import FusedAdam
        net = build(K, 32, train=True)
        dm = net.dyna_module
        with torch.no_grad():
            aff = net.kypt_detector.get_affinity()
        kp = torch.rand(24, 20, K, 4, device="cuda", generator=g) * 1.2 - 0.6
        opt = FusedAdam([p for p in dm.parameters() if p.requires_grad], lr=1e-4)

        def s2():
            opt.zero_grad(set_to_none=True)
            out = dm.encode(kp, aff)
            (out["kypt_recon_loss"] + out["kl_kypt"]).backward()
            opt.step()
        res["stage2_step_ms"] = round(timed(s2, args.iters), 2)
        del net, opt
        print(res, flush=True)


if __name__ == "__main__":
    main()
