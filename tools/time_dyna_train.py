"""Stage-2 timings (training the dynamics module): CUDA events around the eval roll-out (`encode` under no_grad), the
training forward, the backward, the FusedAdam step and the whole step, at the stage-2 shape B = 24, T = 20
(dataset/config.py:26-27) and at B = 1 and B = 96; plus the oracle port's autograd step on the host CPU for one clip.

    python tools/time_dyna_train.py [--iters 20]
"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import nm_oracle as O  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        pl = "unknown"
    return name, pl


def timed(fn, iters):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    import neural_marionette_b200 as nm
    from neural_marionette_b200 import optim
    name, pl = card()
    print(f"card: {name}, power limit {pl}")
    hp = O.default_hparams()
    T, K, S = 20, 24, 10
    for B in (1, 24, 96):
        net = nm.NeuralMarionette(hp)
        net.load_state_dict(O.synthetic_state_dict(hp, seed=7), strict=True)
        net = net.cuda().train()
        dm = net.dyna_module
        with torch.no_grad():
            aff = net.kypt_detector.get_affinity()
        g = torch.Generator().manual_seed(B)
        kp = torch.cat([torch.rand(B, T, K, 3, generator=g) - 0.5, torch.rand(B, T, K, 1, generator=g)], -1).cuda()
        eps = torch.randn(T, S, B, 128, generator=g).cuda()
        opt = optim.FusedAdam(dm.parameters(), lr=4e-4, owner=net)
        state = {}

        def rollout():
            with torch.no_grad():
                dm.encode(kp, aff, eps=eps)

        def fwd():
            out = dm.encode(kp, aff, eps=eps)
            state["loss"] = out["kypt_recon_loss"] + out["kl_kypt"]

        def bwd():
            state["loss"].backward()

        def step():
            opt.zero_grad()
            fwd()
            bwd()
            opt.step()

        for _ in range(3):
            rollout()
            step()
        torch.cuda.synchronize()
        t_roll = timed(rollout, args.iters)
        t_fwd = timed(fwd, args.iters)
        # backward alone: a fresh graph per iteration, built outside the timed window
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        tb = 0.0
        for _ in range(args.iters):
            opt.zero_grad()
            fwd()
            torch.cuda.synchronize()
            ev[0].record()
            bwd()
            ev[1].record()
            torch.cuda.synchronize()
            tb += ev[0].elapsed_time(ev[1])
        t_bwd = tb / args.iters
        t_adam = timed(opt.step, args.iters)
        t_step = timed(step, args.iters)
        print(f"B={B:3d} T={T}: eval roll-out {t_roll:.3f} ms | training forward {t_fwd:.3f} ms | backward {t_bwd:.3f} ms "
              f"({t_bwd / t_roll:.2f}x the roll-out) | FusedAdam step {t_adam:.3f} ms | whole stage-2 step {t_step:.3f} ms")

    # the oracle port's autograd on the host CPU, one clip
    sd = {k: v.clone() for k, v in O.synthetic_state_dict(hp, seed=7).items()}
    leaves = [v.requires_grad_(True) for k, v in sd.items() if k.startswith("dyna_module.") and "offset_param" not in k]
    g = torch.Generator().manual_seed(1)
    kp = torch.cat([torch.rand(1, T, K, 3, generator=g) - 0.5, torch.rand(1, T, K, 1, generator=g)], -1)
    eps = torch.randn(T, S, 1, 128, generator=g)
    skel = O.skeleton_from_affinity(aff.cpu())
    t0 = time.perf_counter()
    out = O.dyna_encode(kp, skel, sd, hp, eps=eps)
    torch.autograd.grad(out["kypt_recon_loss"] + out["kl_kypt"], leaves)
    print(f"oracle port (torch autograd on the host CPU, {os.cpu_count()} threads visible), B=1 T={T}: "
          f"{(time.perf_counter() - t0) * 1e3:.1f} ms forward + backward")


if __name__ == "__main__":
    main()
