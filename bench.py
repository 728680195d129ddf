#!/usr/bin/env python
"""Headline benchmark: voxel frames/sec of keypoint detection (BASELINE.json `metric`).

Workload (`configs[1]`): B = 64 synthetic AIST-shape clips x T = 20 frames x 20 000 points at grid 64^3 per GPU;
one step = fused normalise+voxelize of the raw point clouds + `KyptDetector.forward` (spatio-temporal branch,
per-frame encoder, heat-map head / soft-argmax, decoder, reconstruction BCE and auxiliary losses — what the
reference's forward does).  `value` = frames / second with the raw points resident in HBM; `e2e` = the same
through the public API from pinned host memory (H2D of the points, D2H of the keypoints and the loss inside the
timed region).  Multi-GPU (torchrun): clips shard across ranks, no data-path collective -> weak scaling.

The default line also carries two sub-records measured in the same run, so that the driver's 1/2/4/8-GPU runs see
them: `generate` (configs[2]: `NeuralMarionette.generate`, clips sharded over the ranks) and `train` (configs[3]: the
D-FAUST-shape training step - fwd + bwd + Adam - data-parallel with the NCCL gradient all-reduce over NVLink).
`--workload generate|train` makes one of them the headline of the line instead.

`--dump-outputs DIR` writes what the headline's last timed step returned (rank 0's clips) as DIR/<name>.npy: inputs,
weights and the roll-out noise are seeded, so two builds run with the same arguments can be compared array for array.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload detector|generate|train]
                    [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic conv FLOPs (2*MAC) at G = 64, SURVEY.md §8(d) / BASELINE.md §5
GF_ENC_FRAME, GF_ST_CLIP, GF_DEC_FRAME = 27.848, 93.815, 65.434
METRIC = "voxel frames/sec keypoint detection"
DUMP_BYTES = 64 << 20


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips", type=int, default=None, help="clips per GPU per step (64; 24 for --workload train)")
    ap.add_argument("--frames", type=int, default=None, help="frames per clip (20; 10 for --workload train)")
    ap.add_argument("--points", type=int, default=20000)
    ap.add_argument("--grid", type=int, default=64)
    ap.add_argument("--cpu-baseline-frames", type=int, default=None,
                    help="frames of the ONE clip the CPU arm processes per step (default: a full clip; 3 for train)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the generate / train sub-records of the default line")
    ap.add_argument("--workload", default="detector", choices=["detector", "generate", "train"],
                    help="detector = configs[1] (default, the headline); generate = configs[2] shape "
                         "(NeuralMarionette.generate); train = configs[3] shape (training step, T = 10, 24 clips per GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the arrays the headline's last timed step returned to DIR/<name>.npy (float32 / float64, "
                         f"at most {DUMP_BYTES >> 20} MB in all; larger outputs as a fixed, seeded sample of their elements)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's outputs; it does not apply to --impl reference")
    train = a.workload == "train"
    a.clips = a.clips if a.clips is not None else (24 if train else 64)
    a.frames = a.frames if a.frames is not None else (10 if train else 20)
    a.cpu_baseline_frames = a.cpu_baseline_frames if a.cpu_baseline_frames is not None else (3 if train else a.frames)
    return a


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, source="fallback (B200_PROFILING.md)")


def profiled_traffic(kernel: str, layer: str):
    """dram bytes per launch of the dominant kernel from the committed ncu extract (profiles/roofline_traffic.json:
    {"commit": ..., "entries": [{"kernel", "layer", "dram_bytes_per_frame"}]}).  None when the kernel source changed
    since that profile was taken (the file names the commit it was measured at)."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if not os.path.exists(path):
        return None, None
    try:
        d = json.load(open(path))
        src = os.path.join(ROOT, d.get("source", "neural_marionette_b200/csrc/conv_tc.cu"))
        head = subprocess.run(["git", "-C", ROOT, "log", "-1", "--format=%H", "--", src], capture_output=True, text=True)
        current = head.stdout.strip()
        if current and not current.startswith(d.get("source_commit", "?")[:12]) and not d.get("source_commit", "").startswith(current[:12]):
            return None, f"profile taken at source commit {d.get('source_commit')}, source now at {current[:12]}: stale"
        for e in d["entries"]:
            if e["kernel"] in kernel and e["layer"] == layer:
                return float(e["dram_bytes_per_frame"]), d.get("profile")
    except Exception as exc:  # pragma: no cover
        return None, f"unreadable ({type(exc).__name__})"
    return None, None


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason samples during the timed region (pynvml, 100 ms period)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def synthetic_raw(seed0, B, T, N):
    from oracle import nm_oracle as O   # input generator shared with the tests (not on the measured path)
    base = [O.synthetic_clip(seed0 + b, T, N) for b in range(min(B, 8))]
    rng = np.random.default_rng(seed0)
    out = np.empty((B, T, N, 3), dtype=np.float32)
    for b in range(B):       # 8 distinct clips, re-posed by a random rigid offset/scale: distinct occupancy per clip
        out[b] = base[b % len(base)] * np.float32(rng.uniform(0.8, 1.2)) + rng.uniform(-0.2, 0.2, size=3).astype(np.float32)
    return out


def sample_outputs(out: dict) -> dict:
    """The tensors of a step's result as host arrays (float64 stays float64 and integers become float64, everything else
    float32), DUMP_BYTES at most in all.  An array larger than its equal share of that budget keeps a seeded choice of
    its elements, flattened: the same positions for the same shape, so that two builds compare element for element.
    name -> (full shape, array)."""
    tensors = {k: v.detach() for k, v in sorted(out.items()) if isinstance(v, torch.Tensor)}
    share = DUMP_BYTES // (8 * max(1, len(tensors)))
    res = {}
    for name, t in tensors.items():
        wide = t.dtype == torch.float64 or not (t.dtype.is_floating_point or t.dtype == torch.bool)
        a = t.to(torch.float64 if wide else torch.float32)
        if a.numel() > share:
            pick = np.sort(np.random.default_rng(0).choice(a.numel(), share, replace=False))
            a = a.reshape(-1)[torch.from_numpy(pick).to(a.device)]
        res[name] = (list(t.shape), a.cpu().numpy())
    return res


def write_outputs(path: str, arrays: dict) -> dict:
    os.makedirs(path, exist_ok=True)
    for name, (_, a) in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)
    return {"dir": os.path.abspath(path),
            "arrays": {name: {"shape": shape, "saved": int(a.size)} for name, (shape, a) in arrays.items()}}


# ------------------------------------------------------------------ the CPU arm
def reference_model(grid):
    """The UNMODIFIED reference staged in oracle/_ref by oracle/make_ref.py (build container), with the synthetic
    checkpoint loaded strict=True.  None when it is not there (-> the oracle port)."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    if not os.path.exists(os.path.join(ref, "model", "neural_marionette.py")):
        return None
    import pickle
    from oracle import nm_oracle as O
    sys.path.insert(0, ref)
    try:
        from model.neural_marionette import NeuralMarionette     # the reference's own module
    finally:
        sys.path.remove(ref)
    opt = pickle.load(open(os.path.join(ref, "pretrained", "aist", "opt.pickle"), "rb"))
    opt.grid_size = grid
    net = NeuralMarionette(opt)
    net.load_state_dict(O.synthetic_state_dict(O.default_hparams(grid_size=grid), seed=0), strict=True)
    net.anneal(1)
    return net


def cpu_reference_run(args, steps, warmup, frames):
    """The reference path on the host cores: the reference itself (oracle/_ref) when staged, else the oracle port.
    One step = ONE clip x `frames` frames of the same per-frame work as the GPU arm."""
    import warnings
    from oracle import nm_oracle as O
    from oracle import nm_oracle_grad as OG
    warnings.filterwarnings("ignore")
    torch.set_num_threads(os.cpu_count())
    hp = O.default_hparams(grid_size=args.grid, Tcond=3 if args.workload == "train" else 5)
    sd = O.synthetic_state_dict(hp, seed=0)
    raw = O.synthetic_clip(1000, frames, args.points)
    net = reference_model(args.grid)
    kind = "reference" if net is not None else "port"
    act = {"detector": True, "learner": True}
    opt = None
    if net is not None:
        if args.workload == "train":
            net.train()
            opt = torch.optim.Adam(net.kypt_detector.parameters(), lr=4e-4)     # train.py:380, dataset/config.py:12
        else:
            net.eval()
            if args.workload == "generate":
                net.Tcond = hp.Tcond
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        vox = torch.from_numpy(O.voxelize_clip(O.episodic_normalization(raw), args.grid))[None]
        if args.workload == "train":
            if net is not None:
                opt.zero_grad()
                loss = OG.detector_loss(net.kypt_detector(vox), recon_only=False)
                loss.backward()
                opt.step()
            else:
                OG.detector_gradients(vox, sd, hp, recon_only=False)
        else:
            with torch.no_grad():
                if args.workload == "generate":
                    if net is not None:
                        if i == 0:
                            net(vox, act)                   # builds the skeleton once, as the reference requires
                        float(net.generate(vox, act)["gen"][:, -1].mean())
                    else:
                        float(O.marionette_generate(vox, sd, hp)["gen"][:, -1].mean())
                elif net is not None:
                    float(net.kypt_detector(vox)["recon_loss"])
                else:
                    float(O.detector_forward(vox, sd, hp)["recon_loss"])
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = float(np.mean(times))
    return frames / t, t, torch.get_num_threads(), kind


def workload_text(args, B, T, N, G, world):
    if args.workload == "generate":
        return (f"NeuralMarionette.generate (voxelize + detector on Tcond=5 frames + {T}-step HSVRNN roll-out + decode of "
                f"the {T - 5} generated frames) on {B} synthetic clips x {T} frames x {N} pts per GPU, grid {G}^3, K=24")
    if args.workload == "train":
        return (f"training step (voxelize + KyptDetector fwd + bwd of the stage-1 loss sum + Adam; NCCL gradient all-reduce "
                f"x{world}) on {B} synthetic D-FAUST-shape clips x {T} frames x {N} pts per GPU, grid {G}^3, K=24")
    return (f"KyptDetector.forward (voxelize + ST branch + encoder + head/soft-argmax + decoder + losses) "
            f"on {B} synthetic AIST-shape clips x {T} frames x {N} pts per GPU, grid {G}^3, K=24")


def reference_arm(args):
    """`--impl reference`: the reference's CPU implementation of the workload on this box's host cores.  The line reports
    exactly what ran: `steps` / `warmup` executed and the ONE-clip sample each step processes."""
    frames = max(2, args.cpu_baseline_frames)
    steps, warmup = args.steps, max(1, min(args.warmup, 2))
    fps, t, cores, kind = cpu_reference_run(args, steps, warmup, frames)
    what = {"detector": "KyptDetector.forward", "generate": "NeuralMarionette.generate",
            "train": "KyptDetector fwd + bwd + Adam"}[args.workload]
    sample = (f"1 clip x {frames} frames x {args.points} pts per step (voxelize + {what}), {warmup} warm-up + {steps} timed "
              f"steps of {t:.2f} s; same per-frame work as the GPU arm's {args.clips}-clip steps")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmup, "steps_requested": args.steps, "warmup_requested": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_text(args, 1, frames, args.points, args.grid, 1) + " [CPU arm: ONE clip per step]",
                   "clips_per_step": 1, "frames_per_clip": frames, "points_per_frame": args.points, "grid": args.grid,
                   "gpu_arm_workload": workload_text(args, args.clips, args.frames, args.points, args.grid, args.gpus)},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------ the GPU arm
class HostFeed:
    """The end-to-end leg's input pipeline, as a training / serving loop would write it: the step's points live in pinned
    host memory and are copied to the device EVERY step (inside the timed region) on a copy stream, double-buffered so
    that the copy for step k+1 runs while step k computes.  `next()` returns step k's device tensor (the compute stream
    waits for its copy) and starts the copy for step k+1; the result read-back is pinned + asynchronous the same way."""

    def __init__(self, host: torch.Tensor, dev):
        self.host, self.dev = host, dev
        self.stream = torch.cuda.Stream(device=dev)
        self.buf = [torch.empty(host.shape, dtype=host.dtype, device=dev) for _ in range(2)]
        self.done = [torch.cuda.Event(), torch.cuda.Event()]
        self.i, self.primed = 0, False

    def _issue(self, slot):
        cur = torch.cuda.current_stream(self.dev)
        self.stream.wait_stream(cur)                    # the slot's previous reader (two steps ago) has been enqueued before
        with torch.cuda.stream(self.stream):
            self.buf[slot].copy_(self.host, non_blocking=True)
            self.done[slot].record(self.stream)

    def next(self) -> torch.Tensor:
        cur = torch.cuda.current_stream(self.dev)
        if not self.primed:
            self._issue(self.i)
            self.primed = True
        cur.wait_event(self.done[self.i])
        x = self.buf[self.i]
        self.i ^= 1
        self._issue(self.i)
        return x


class Bench:
    def __init__(self, args):
        import torch.distributed as dist
        import neural_marionette_b200 as nm
        from neural_marionette_b200 import _lib, ops
        from oracle import nm_oracle as O   # synthetic weights / inputs and the cpu_baseline leg only
        self.args, self.dist, self.nm, self.lib, self.ops, self.O = args, dist, nm, _lib, ops, O
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm"
        torch.manual_seed(0)                # the roll-out noise of `generate`: the same every run
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        _lib.call("nm_device_supported")
        self.G = args.grid
        self.training_profile = False

    def model(self, Tcond=5):
        hp = self.O.default_hparams(grid_size=self.G, Tcond=Tcond)
        net = self.nm.NeuralMarionette(hp)
        net.load_state_dict(self.O.synthetic_state_dict(hp, seed=0), strict=True)
        net = net.to(self.dev)
        net.anneal(1)
        return net, hp

    def timed(self, fn, steps, keep_last=False):
        """Device time per call of `fn` over `steps` calls (slowest rank); with keep_last, (time, what the last call
        returned)."""
        from neural_marionette_b200.parallel import barrier, max_over_ranks
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()
        e1.record()
        barrier()
        ms = max_over_ranks(e0.elapsed_time(e1), self.dev) / steps      # device time, slowest rank
        return (ms, last) if keep_last else ms

    # ---- configs[1] / configs[2]: inference
    def run_inference(self, workload, B, T, N, steps, warmup, want_roofline, keep_outputs=False):
        ops, G, dev = self.ops, self.G, self.dev
        net, hp = self.model()
        net.eval()
        det = net.kypt_detector
        raw_host = torch.from_numpy(synthetic_raw(1000 + 100 * self.rank, B, T, N)).pin_memory()
        raw_dev = raw_host.to(dev)
        feed = HostFeed(raw_host, dev)
        act = {"detector": True, "learner": True}
        if workload == "generate":
            with torch.no_grad():
                net(ops.normalize_voxelize(raw_dev[:2], G, check=False), act)   # builds the skeleton once, as the reference requires

            def step_resident():
                return net.generate(ops.normalize_voxelize(raw_dev, G, check=False), act)

            def step_e2e():
                out = net.generate(ops.normalize_voxelize(feed.next(), G, check=False), act)
                return out["keypoints"].cpu(), float(out["gen"][:, -1].mean())
        else:
            def step_resident():
                return det(ops.normalize_voxelize(raw_dev, G, check=False))

            def step_e2e():
                out = det(ops.normalize_voxelize(feed.next(), G, check=False))
                return out["keypoints"].cpu(), float(out["recon_loss"])
        res = {}
        with torch.no_grad():
            for _ in range(warmup):
                step_resident()
            sampler = ClockSampler(self.local)
            sampler.start()
            calls0 = self.lib.CALLS
            ops.PROFILE = {} if want_roofline else None
            ms, out = self.timed(step_resident, steps, keep_last=True)
            prof, ops.PROFILE = ops.PROFILE, None
            res["launches"] = self.lib.CALLS - calls0
            res["clocks"] = sampler.result()
            res["outputs"] = sample_outputs(out) if keep_outputs else None
            del out
            step_e2e()
            ms_e2e = self.timed(step_e2e, steps)
            if workload == "detector" and want_roofline:
                # SURVEY.md §8(d) config #2 asks for the encoder-only figure next to the full forward
                def step_encoder():
                    return det.vox_to_kypt(ops.normalize_voxelize(raw_dev, G, check=False))
                step_encoder()
                ms_enc = self.timed(step_encoder, steps)
                res["encoder_only"] = {
                    "value": self.world * B * T / (ms_enc / 1e3), "unit": "frames/s", "ms_per_step": ms_enc,
                    "workload": "voxelize + VoxToKyptNet.forward (no decoder, no losses), same clips",
                    "model_tflops": self.world * B * (GF_ST_CLIP + T * GF_ENC_FRAME) / (ms_enc / 1e3) / 1e3 if G == 64 else None}
        frames_total = self.world * B * T
        res.update(ms=ms, ms_e2e=ms_e2e, value=frames_total / (ms / 1e3), e2e=frames_total / (ms_e2e / 1e3),
                   h2d=int(raw_host.numel() * 4), d2h=int(B * T * 24 * 4 * 4 + 4), prof=prof, hp=hp)
        if G == 64:
            gf = B * (GF_ST_CLIP + T * (GF_ENC_FRAME + GF_DEC_FRAME)) if workload == "detector" else \
                B * (GF_ST_CLIP + hp.Tcond * (GF_ENC_FRAME + GF_DEC_FRAME) + (T - hp.Tcond) * GF_DEC_FRAME)
            res["model_tflops"] = self.world * gf / (ms / 1e3) / 1e3
        del net
        torch.cuda.empty_cache()
        return res

    # ---- configs[3]: the training step
    def run_train(self, B, T, N, steps, warmup, keep_outputs=False):
        """fwd + bwd of the stage-1 loss sum (train.py:173-181 weights) + Adam (train.py:380-409) on B clips x T frames
        per GPU (dataset/config.py:4-12: T = 10, batch 24); gradients all-reduced over the ranks in 4 buckets launched
        from the backward (parallel.GradientBuckets, NCCL)."""
        from oracle import nm_oracle_grad as OG         # only the loss weights of train.py:68-78 (a dict)
        from neural_marionette_b200 import optim
        ops, G, dev = self.ops, self.G, self.dev
        net, hp = self.model(Tcond=3)
        net.train()
        det = net.kypt_detector
        opt = optim.FusedAdam(det.parameters(), lr=4e-4, owner=net)
        raw_host = torch.from_numpy(synthetic_raw(2000 + 100 * self.rank, B, T, N)).pin_memory()
        raw_dev = raw_host.to(dev)
        ev = {"finish": []}

        feed = HostFeed(raw_host, dev)

        def step(src):
            vox = ops.normalize_voxelize(src if src.is_cuda else feed.next(), G, check=False)
            opt.zero_grad()
            out = det(vox)
            loss = OG.detector_loss(out, recon_only=False)
            loss.backward()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            opt.buckets.finish()                        # waits for the bucketed all-reduce (already in flight)
            b.record()
            ev["finish"].append((a, b))
            opt.step()
            return out

        for _ in range(warmup):
            step(raw_dev)
        torch.cuda.reset_peak_memory_stats()
        ev["finish"].clear()
        sampler = ClockSampler(self.local)
        sampler.start()
        calls0 = self.lib.CALLS
        ms, out = self.timed(lambda: step(raw_dev), steps, keep_last=True)
        launches = self.lib.CALLS - calls0
        clocks = sampler.result()
        torch.cuda.synchronize()
        outputs = sample_outputs(out) if keep_outputs else None
        del out
        # per-launch CUDA events of the tensor-core convs / weight gradients over two more steps (kept out of `ms`)
        ops.PROFILE = {}
        prof_ms = self.timed(lambda: step(raw_dev), 2)
        prof, ops.PROFILE = ops.PROFILE, None
        exposed = float(np.mean([a.elapsed_time(b) for a, b in ev["finish"]]))
        ms_e2e = self.timed(lambda: float(step(raw_host)["recon_loss"].detach()), steps)
        # the all-reduce on its own (no overlap): the 4 buckets back to back on an idle GPU
        ar_ms = None
        if self.world > 1:
            flat = opt.buckets.flat
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            self.dist.barrier()
            a.record()
            for _ in range(5):
                for lo, hi in opt.buckets.bounds:
                    self.dist.all_reduce(flat[lo:hi])
            b.record()
            torch.cuda.synchronize()
            ar_ms = a.elapsed_time(b) / 5
        frames_total = self.world * B * T
        # the same step captured in ONE CUDA graph and replayed (single rank: the NCCL exchange is driven from Python hooks);
        # same launches, bit-identical results (tests/test_gpu_backward.py::test_captured_training_step_matches_eager)
        graph_rec = None
        if self.world == 1 and os.environ.get("NM_BENCH_TRAIN_GRAPH", "1") != "0":
            from neural_marionette_b200 import graph as nm_graph
            try:
                cap = nm_graph.CapturedTrainStep(det, opt, lambda out: OG.detector_loss(out, recon_only=False), raw_dev, G, warmup=2)
                g_ms = self.timed(lambda: cap(raw_dev), steps)
                g_e2e = self.timed(lambda: float(cap(feed.next())), steps)
                opt.sync_counters()
                graph_rec = {"value": frames_total / (g_ms / 1e3), "unit": "frames/s", "ms_per_step": g_ms,
                             "e2e": {"value": frames_total / (g_e2e / 1e3), "unit": "frames/s", "ms_per_step": g_e2e},
                             "note": "graph.CapturedTrainStep: normalise + voxelize, forward, backward and the device-side Adam "
                                     "step replayed as one CUDA graph; e2e adds the H2D copy of the points and the D2H read of "
                                     "the loss every step"}
            except Exception as e:      # report, do not hide: the eager numbers above stand on their own
                graph_rec = {"error": f"{type(e).__name__}: {e}"[:300]}
        res = dict(ms=ms, ms_e2e=ms_e2e, value=frames_total / (ms / 1e3), e2e=frames_total / (ms_e2e / 1e3), graph=graph_rec,
                   h2d=int(raw_host.numel() * 4), d2h=4, launches=launches,
                   grad_bytes=int(opt.buckets.flat.numel() * 4), buckets=len(opt.buckets.bounds), exposed_ms=exposed,
                   allreduce_alone_ms=ar_ms, skipped=opt.skipped, peak_gib=torch.cuda.max_memory_allocated() / 2 ** 30,
                   grad_scale=ops.grad_scale(), clocks=clocks, prof=prof, prof_ms=prof_ms, outputs=outputs)
        if G == 64:   # training ~ 3x the forward's conv FLOPs (fwd + dgrad + wgrad)
            res["model_tflops"] = 3 * self.world * B * (GF_ST_CLIP + T * (GF_ENC_FRAME + GF_DEC_FRAME)) / (ms / 1e3) / 1e3
        del net, opt
        torch.cuda.empty_cache()
        return res

    def train_record(self, r, B, T):
        rec = {"value": r["value"], "unit": "frames/s", "ms_per_step": r["ms"],
               "workload": f"training step (fwd + bwd + Adam), {B} clips x {T} frames per GPU, grid {self.G}^3; stage-1 loss sum",
               "e2e": {"value": r["e2e"], "unit": "frames/s", "ms_per_step": r["ms_e2e"], "h2d_bytes_per_step": r["h2d"],
                       "d2h_bytes_per_step": r["d2h"]},
               "model_tflops": r.get("model_tflops"), "gpu_launches": int(r["launches"]),
               "allreduce": {"backend": "nccl" if self.world > 1 else "none (1 rank)", "ranks": self.world,
                             "bytes": r["grad_bytes"], "buckets": r["buckets"],
                             "exposed_ms_per_step": r["exposed_ms"], "alone_ms": r["allreduce_alone_ms"],
                             "note": "buckets are all-reduced asynchronously from post-accumulate hooks while the rest of the "
                                     "backward runs; exposed = device time spent waiting for them after the backward"},
               "skipped_steps": r["skipped"], "peak_memory_gib": r["peak_gib"], "loss_scale": r["grad_scale"]}
        if r.get("graph") is not None:
            rec["cuda_graph"] = r["graph"]
        return rec

    def roofline(self, prof, ms, steps):
        pk = peaks()
        torch.cuda.synchronize()
        by_shape = {}
        for key, evs in (prof or {}).items():
            by_shape[key] = (sum(a.elapsed_time(b) for a, b in evs), len(evs))
        if not by_shape:
            return None
        tot_ms = sum(v[0] for v in by_shape.values())
        tot_flop = sum(k[-1] * v[1] for k, v in by_shape.items())
        (kind, tn, tD, tci, tco, tk, ts, tflop), (t_ms, cnt) = max(by_shape.items(), key=lambda kv: kv[1][0])
        ach = tflop * cnt / (t_ms / 1e3) / 1e12
        slab3 = tk == 3 and ts == 1 and tD % 16 == 0 and tci in (32, 64, 128) and tco <= 128 and \
            tco % (32 if tci <= 64 else 16) == 0
        kernel = "conv_wgrad_tc_kernel" if kind == "wgrad" else ("conv3d_slab3_kernel" if slab3 else "conv3d_tc_kernel")
        layer = f"grid={tD} Cin={tci} Cout={tco} k={tk} s={ts}"
        per_frame, src = profiled_traffic(kernel, layer)
        entry = "nm_conv3d_k3_wgrad_tc, tcgen05 weight gradient" if kind == "wgrad" else "nm_conv3d_tc, tcgen05 implicit GEMM"
        return {"bound": "tensor", "kernel": f"{kernel} ({entry})",
                "layer": f"n={tn} " + layer, "achieved": ach, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sust"],
                "traffic": per_frame * tn if per_frame is not None else None, "traffic_source": src,
                "note": "dec.8: conv3d_k3(upsample2x(LeakyReLU(GroupNorm(x)))) in one kernel; FLOPs counted are the "
                        "conv's only" if (kind, tD, tci, tco, tk) == ("conv", 64, 64, 32, 3) and not self.training_profile else
                        ("forward convs and data gradients (the same kernels on mirrored weights) share a shape key" if
                         self.training_profile and kind == "conv" else None),
                "peak_source": pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)",
                "launch_ms": t_ms / cnt, "share_of_step": t_ms / (ms * steps),
                "all_tc_convs": {"achieved": tot_flop / (tot_ms / 1e3) / 1e12, "share_of_step": tot_ms / (ms * steps)},
                "by_layer": [{"layer": f"{k[0]} n={k[1]} grid={k[2]} {k[3]}->{k[4]} k{k[5]}s{k[6]}", "launches": v[1],
                              "ms_per_launch": round(v[0] / v[1], 4),
                              "tflops": round(k[7] * v[1] / (v[0] / 1e3) / 1e12, 1),
                              "share_of_step": round(v[0] / (ms * steps), 4)}
                             for k, v in sorted(by_shape.items(), key=lambda kv: -kv[1][0])[:30]]}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        if rank == 0:
            reference_arm(args)
        return
    be = Bench(args)
    B, T, N, G = args.clips, args.frames, args.points, args.grid
    steps, warmup = args.steps, max(3, args.warmup)
    config = {"workload": workload_text(args, B, T, N, G, world), "clips_per_gpu": B, "frames_per_clip": T,
              "points_per_frame": N, "grid": G,
              "l2": "inputs (points + >20 GB of activations per step) exceed the 126 MB L2",
              "precision": "fp16 activations/weights at rest, fp32 accumulation (tcgen05 kind::f16), fp32 GroupNorm "
                           "statistics / heads / losses" + ("; fp16 loss-scaled activation gradients, fp32 parameter "
                                                            "gradients and Adam state" if args.workload == "train" else ""),
              "parallelism": f"clip-sharded x{world}, " + ("NCCL gradient all-reduce (4 buckets, overlapped with the backward)"
                                                          if args.workload == "train" else "no data-path collective")}
    line = {"metric": METRIC, "unit": "frames/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": config}
    dump = args.dump_outputs is not None
    if args.workload == "train":
        r = be.run_train(B, T, N, steps, warmup, keep_outputs=dump)
        rec = be.train_record(r, B, T)
        be.training_profile = True
        line.update(value=r["value"], ms_per_step=r["ms"], e2e=rec["e2e"], gpu_launches=int(r["launches"]),
                    model_tflops=r.get("model_tflops"), train=rec, roofline=be.roofline(r["prof"], r["prof_ms"], 2),
                    clocks=r["clocks"])
        line["e2e"]["note"] = "host points -> device every step; the step's loss read back"
    else:
        r = be.run_inference(args.workload, B, T, N, steps, warmup, want_roofline=True, keep_outputs=dump)
        line.update(value=r["value"], ms_per_step=r["ms"], clocks=r["clocks"],
                    e2e={"value": r["e2e"], "unit": "frames/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                         "ms_per_step": r["ms_e2e"],
                         "note": "H2D = the step's raw points from pinned host memory, every step, on a copy stream "
                                 "(double-buffered: the copy of step k+1 overlaps step k); D2H = the keypoints (B, T, 24, 4) "
                                 "+ the loss scalar: the result of a keypoint-detection step; the reconstruction volumes "
                                 "stay on the device"},
                    gpu_launches=int(r["launches"]),
                    gpu_launches_note="C-ABI calls inside the timed region (each enqueues >= 1 of our kernels)",
                    model_tflops=r.get("model_tflops"), roofline=be.roofline(r["prof"], r["ms"], steps))
        if "encoder_only" in r:
            line["encoder_only"] = r["encoder_only"]
        if args.workload == "detector" and not args.no_sub:
            sub_steps = max(2, min(steps, 5))
            g = be.run_inference("generate", B, T, N, sub_steps, 3, want_roofline=False)
            line["generate"] = {"value": g["value"], "unit": "frames/s", "ms_per_step": g["ms"], "steps": sub_steps,
                                "workload": f"configs[2]: NeuralMarionette.generate, {B} clips x {T} frames per GPU (Tcond 5), "
                                            f"clips sharded x{world}",
                                "e2e": {"value": g["e2e"], "unit": "frames/s", "ms_per_step": g["ms_e2e"]},
                                "model_tflops": g.get("model_tflops"), "gpu_launches": int(g["launches"])}
            tr = be.run_train(24, 10, N, sub_steps, 3)
            line["train"] = dict(be.train_record(tr, 24, 10), steps=sub_steps)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        fps, t, cores, kind = cpu_reference_run(args, 2, 1, args.cpu_baseline_frames)
        line["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": kind,
                                "sample": f"1 clip x {args.cpu_baseline_frames} frames (voxelize + {args.workload}), "
                                          f"1 warm-up + 2 timed reps of {t:.1f} s; same per-frame work as the GPU arm"}
    if rank == 0 and dump:
        line["outputs"] = write_outputs(args.dump_outputs, r["outputs"])
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        be.dist.destroy_process_group()


if __name__ == "__main__":
    main()
