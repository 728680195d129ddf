"""Device time of the HSVRNN roll-out (5 conditioned + 15 generated steps) at several batch sizes (the cluster kernel
serves B <= 96, the one-CTA-per-element kernel B = 256): CUDA events around `HSVRNNBVH.generate`, and the same
roll-out replayed as a CUDA graph (what a latency-bound caller would do; the draws are injected so the graph is static)."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import neural_marionette_b200 as nm          # noqa: E402
from oracle import nm_oracle as O            # synthetic weights only  # noqa: E402

hp = O.default_hparams(grid_size=32)
net = nm.NeuralMarionette(hp)
net.load_state_dict(O.synthetic_state_dict(hp, 0))
net = net.cuda().eval()
net.anneal(1)
dyn = net.dyna_module
g = torch.Generator(device="cuda").manual_seed(0)
for B in (1, 4, 16, 64, 256):
    kp = torch.rand(B, 5, 24, 4, device="cuda", generator=g) * 1.2 - 0.6
    with torch.no_grad():
        dyn.encode(kp, net.kypt_detector.get_affinity())                      # builds the skeleton
        ec = torch.randn(5, 10, B, 128, device="cuda", generator=g)
        eg = torch.randn(15, B, 128, device="cuda", generator=g)
        run = lambda: dyn.generate(kp, None, Ttot=20, Tcond=5, eps_cond=ec, eps_gen=eg)   # noqa: E731
        for _ in range(3):
            run()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for _ in range(10):
            run()
        b.record()
        torch.cuda.synchronize()
        eager = a.elapsed_time(b) / 10
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            run()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=s):
                out = run()
        torch.cuda.synchronize()
        a.record()
        for _ in range(20):
            gr.replay()
        b.record()
        torch.cuda.synchronize()
        print(f"B={B:4d}: 20-step roll-out eager {eager:.3f} ms, CUDA-graph replay {a.elapsed_time(b) / 20:.3f} ms "
              f"({a.elapsed_time(b) / 20 / 20 * 1e3:.1f} us per step)")
