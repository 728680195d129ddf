"""The stage-1 training step's backward kernels at the size the step runs: 24 clips x 10 frames at grid 64^3 with 24
keypoints, all 240 frames in one pass (`bench.py --workload train`).  There the decoder's 64-channel 64^3 tensors hold
4.03e9 elements (8.05 GB, past 2^31 elements and 2^32 bytes) and every 32-channel 64^3 tensor 2.01e9 (past 2^31 bytes).

A float64 backward of the whole batch is out of reach, so every full-size input is built on the device from D = 3
distinct samples (frames, or clips where a kernel couples a clip's frames) by an owner map (`owner_map`):
  1. copy identity: every copy of an owner is bit-identical to its first copy - this reads every byte of the output,
     past 2^31 and 2^32 included;
  2. float64 reference of the D distinct samples: a per-sample output against the reference of its owner, a
     batch-reduced output (weight / bias / GroupNorm / head gradients) against sum_d m_d ref_d, m_d = copies of d;
  3. bounds relative to the largest reference entry, from fp16 operands and fp32 accumulation (measured errors printed).

`STEP_SHAPES` lists every (backward entry point, shape) one real step runs (`test_step_shapes_are_all_listed` keeps it
complete).  Run as a script on a GPU (`PYTHONPATH=. python tests/test_gpu_train_scale.py`), this file prints that list."""
import copy
import gc
import time

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import nm_oracle as O
from oracle import nm_oracle_grad as OG

gpu = pytest.mark.gpu

G, B, T, K, ND = 64, 24, 10, 24, 3          # the step's grid, clips, frames per clip, keypoints; distinct samples

# (entry point of `ops`, shape key) of one 24 x 10 step at G = 64, K = 24 - see `_shape_key` for what a key holds
STEP_SHAPES = [
    ('chamfer_vol_fit_backward', (240, 64, 64, 64, 24)),
    ('conv3d_input_grad', (24, 2, 2, 2, 48, 48, 2, 2)),
    ('conv3d_input_grad', (24, 2, 2, 2, 72, 48, 1, 1)),
    ('conv3d_input_grad', (24, 2, 2, 2, 72, 48, 3, 1)),
    ('conv3d_input_grad', (24, 2, 2, 2, 72, 72, 3, 1)),
    ('conv3d_input_grad', (24, 4, 4, 4, 32, 32, 2, 2)),
    ('conv3d_input_grad', (24, 4, 4, 4, 48, 32, 1, 1)),
    ('conv3d_input_grad', (24, 4, 4, 4, 48, 32, 3, 1)),
    ('conv3d_input_grad', (24, 4, 4, 4, 48, 48, 3, 1)),
    ('conv3d_input_grad', (24, 8, 8, 8, 32, 32, 3, 1)),
    ('conv3d_input_grad', (24, 8, 8, 8, 32, 128, 1, 1)),
    ('conv3d_input_grad', (24, 8, 8, 8, 32, 128, 3, 1)),
    ('conv3d_input_grad', (24, 8, 8, 8, 128, 128, 2, 2)),
    ('conv3d_input_grad', (24, 16, 16, 16, 128, 128, 2, 2)),
    ('conv3d_input_grad', (24, 16, 16, 16, 128, 128, 3, 1)),
    ('conv3d_input_grad', (24, 16, 16, 16, 256, 128, 1, 1)),
    ('conv3d_input_grad', (24, 16, 16, 16, 256, 128, 3, 1)),
    ('conv3d_input_grad', (24, 16, 16, 16, 256, 256, 3, 1)),
    ('conv3d_input_grad', (24, 32, 32, 32, 64, 64, 2, 2)),
    ('conv3d_input_grad', (24, 32, 32, 32, 128, 64, 1, 1)),
    ('conv3d_input_grad', (24, 32, 32, 32, 128, 64, 3, 1)),
    ('conv3d_input_grad', (24, 32, 32, 32, 128, 128, 3, 1)),
    ('conv3d_input_grad', (240, 2, 2, 2, 48, 48, 2, 2)),
    ('conv3d_input_grad', (240, 2, 2, 2, 72, 48, 1, 1)),
    ('conv3d_input_grad', (240, 2, 2, 2, 72, 48, 3, 1)),
    ('conv3d_input_grad', (240, 2, 2, 2, 72, 72, 3, 1)),
    ('conv3d_input_grad', (240, 4, 4, 4, 32, 32, 2, 2)),
    ('conv3d_input_grad', (240, 4, 4, 4, 48, 32, 1, 1)),
    ('conv3d_input_grad', (240, 4, 4, 4, 48, 32, 3, 1)),
    ('conv3d_input_grad', (240, 4, 4, 4, 48, 48, 3, 1)),
    ('conv3d_input_grad', (240, 8, 8, 8, 32, 32, 3, 1)),
    ('conv3d_input_grad', (240, 8, 8, 8, 32, 64, 1, 1)),
    ('conv3d_input_grad', (240, 8, 8, 8, 32, 64, 3, 1)),
    ('conv3d_input_grad', (240, 8, 8, 8, 64, 64, 2, 2)),
    ('conv3d_input_grad', (240, 16, 16, 16, 64, 64, 2, 2)),
    ('conv3d_input_grad', (240, 16, 16, 16, 64, 64, 3, 1)),
    ('conv3d_input_grad', (240, 16, 16, 16, 128, 64, 1, 1)),
    ('conv3d_input_grad', (240, 16, 16, 16, 128, 64, 3, 1)),
    ('conv3d_input_grad', (240, 16, 16, 16, 128, 128, 3, 1)),
    ('conv3d_input_grad', (240, 32, 32, 32, 32, 32, 2, 2)),
    ('conv3d_input_grad', (240, 32, 32, 32, 64, 32, 1, 1)),
    ('conv3d_input_grad', (240, 32, 32, 32, 64, 32, 3, 1)),
    ('conv3d_input_grad', (240, 32, 32, 32, 64, 64, 3, 1)),
    ('conv3d_input_grad', (240, 32, 32, 32, 64, 128, 3, 1)),
    ('conv3d_input_grad', (240, 64, 64, 64, 32, 32, 3, 1)),
    ('conv3d_input_grad', (240, 64, 64, 64, 32, 64, 3, 1)),
    ('conv3d_weight_grad', (24, 2, 2, 2, 48, 72, 1, 1)),
    ('conv3d_weight_grad', (24, 2, 2, 2, 48, 72, 3, 1)),
    ('conv3d_weight_grad', (24, 2, 2, 2, 72, 72, 3, 1)),
    ('conv3d_weight_grad', (24, 4, 4, 4, 32, 48, 1, 1)),
    ('conv3d_weight_grad', (24, 4, 4, 4, 32, 48, 3, 1)),
    ('conv3d_weight_grad', (24, 4, 4, 4, 48, 48, 2, 2)),
    ('conv3d_weight_grad', (24, 4, 4, 4, 48, 48, 3, 1)),
    ('conv3d_weight_grad', (24, 8, 8, 8, 32, 32, 2, 2)),
    ('conv3d_weight_grad', (24, 8, 8, 8, 32, 32, 3, 1)),
    ('conv3d_weight_grad', (24, 8, 8, 8, 128, 32, 1, 1)),
    ('conv3d_weight_grad', (24, 8, 8, 8, 128, 32, 3, 1)),
    ('conv3d_weight_grad', (24, 16, 16, 16, 128, 128, 2, 2)),
    ('conv3d_weight_grad', (24, 16, 16, 16, 128, 128, 3, 1)),
    ('conv3d_weight_grad', (24, 16, 16, 16, 128, 256, 1, 1)),
    ('conv3d_weight_grad', (24, 16, 16, 16, 128, 256, 3, 1)),
    ('conv3d_weight_grad', (24, 16, 16, 16, 256, 256, 3, 1)),
    ('conv3d_weight_grad', (24, 32, 32, 32, 64, 128, 1, 1)),
    ('conv3d_weight_grad', (24, 32, 32, 32, 64, 128, 3, 1)),
    ('conv3d_weight_grad', (24, 32, 32, 32, 128, 128, 2, 2)),
    ('conv3d_weight_grad', (24, 32, 32, 32, 128, 128, 3, 1)),
    ('conv3d_weight_grad', (24, 64, 64, 64, 64, 64, 2, 2)),
    ('conv3d_weight_grad', (240, 2, 2, 2, 48, 72, 1, 1)),
    ('conv3d_weight_grad', (240, 2, 2, 2, 48, 72, 3, 1)),
    ('conv3d_weight_grad', (240, 2, 2, 2, 72, 72, 3, 1)),
    ('conv3d_weight_grad', (240, 4, 4, 4, 32, 48, 1, 1)),
    ('conv3d_weight_grad', (240, 4, 4, 4, 32, 48, 3, 1)),
    ('conv3d_weight_grad', (240, 4, 4, 4, 48, 48, 2, 2)),
    ('conv3d_weight_grad', (240, 4, 4, 4, 48, 48, 3, 1)),
    ('conv3d_weight_grad', (240, 8, 8, 8, 32, 32, 2, 2)),
    ('conv3d_weight_grad', (240, 8, 8, 8, 32, 32, 3, 1)),
    ('conv3d_weight_grad', (240, 8, 8, 8, 64, 32, 1, 1)),
    ('conv3d_weight_grad', (240, 8, 8, 8, 64, 32, 3, 1)),
    ('conv3d_weight_grad', (240, 16, 16, 16, 64, 64, 2, 2)),
    ('conv3d_weight_grad', (240, 16, 16, 16, 64, 64, 3, 1)),
    ('conv3d_weight_grad', (240, 16, 16, 16, 64, 128, 1, 1)),
    ('conv3d_weight_grad', (240, 16, 16, 16, 64, 128, 3, 1)),
    ('conv3d_weight_grad', (240, 16, 16, 16, 128, 128, 3, 1)),
    ('conv3d_weight_grad', (240, 32, 32, 32, 32, 64, 1, 1)),
    ('conv3d_weight_grad', (240, 32, 32, 32, 32, 64, 3, 1)),
    ('conv3d_weight_grad', (240, 32, 32, 32, 64, 64, 2, 2)),
    ('conv3d_weight_grad', (240, 32, 32, 32, 64, 64, 3, 1)),
    ('conv3d_weight_grad', (240, 32, 32, 32, 128, 64, 3, 1)),
    ('conv3d_weight_grad', (240, 64, 64, 64, 32, 32, 2, 2)),
    ('conv3d_weight_grad', (240, 64, 64, 64, 32, 32, 3, 1)),
    ('conv3d_weight_grad', (240, 64, 64, 64, 64, 32, 3, 1)),
    ('conv_transpose3d_input_grad', (24, 4, 4, 4, 48, 72)),
    ('conv_transpose3d_input_grad', (24, 8, 8, 8, 32, 48)),
    ('conv_transpose3d_input_grad', (24, 16, 16, 16, 128, 32)),
    ('conv_transpose3d_input_grad', (240, 4, 4, 4, 48, 72)),
    ('conv_transpose3d_input_grad', (240, 8, 8, 8, 32, 48)),
    ('conv_transpose3d_input_grad', (240, 16, 16, 16, 64, 32)),
    ('conv_transpose3d_weight_grad', (24, 2, 2, 2, 72, 48)),
    ('conv_transpose3d_weight_grad', (24, 4, 4, 4, 48, 32)),
    ('conv_transpose3d_weight_grad', (24, 8, 8, 8, 32, 128)),
    ('conv_transpose3d_weight_grad', (240, 2, 2, 2, 72, 48)),
    ('conv_transpose3d_weight_grad', (240, 4, 4, 4, 48, 32)),
    ('conv_transpose3d_weight_grad', (240, 8, 8, 8, 32, 64)),
    ('decoder_adjust_backward', (24, 16, 16, 16, 128, 10, 16, 24)),
    ('final_recon_backward_fused', (240, 64, 64, 64, 32)),
    ('first_conv_weight_grad', (24, 64, 64, 64, 64)),
    ('first_conv_weight_grad', (240, 64, 64, 64, 32)),
    ('groupnorm_backward', (24, 2, 2, 2, 48, 3, 1, 1)),
    ('groupnorm_backward', (24, 2, 2, 2, 72, 4, 0, 1)),
    ('groupnorm_backward', (24, 2, 2, 2, 72, 4, 1, 1)),
    ('groupnorm_backward', (24, 4, 4, 4, 32, 2, 1, 1)),
    ('groupnorm_backward', (24, 4, 4, 4, 48, 3, 0, 1)),
    ('groupnorm_backward', (24, 4, 4, 4, 48, 3, 1, 1)),
    ('groupnorm_backward', (24, 8, 8, 8, 32, 2, 0, 1)),
    ('groupnorm_backward', (24, 8, 8, 8, 32, 2, 1, 1)),
    ('groupnorm_backward', (24, 8, 8, 8, 128, 8, 1, 1)),
    ('groupnorm_backward', (24, 16, 16, 16, 128, 8, 0, 1)),
    ('groupnorm_backward', (24, 16, 16, 16, 128, 8, 1, 1)),
    ('groupnorm_backward', (24, 16, 16, 16, 256, 16, 0, 1)),
    ('groupnorm_backward', (24, 16, 16, 16, 256, 16, 1, 1)),
    ('groupnorm_backward', (24, 32, 32, 32, 64, 4, 1, 1)),
    ('groupnorm_backward', (24, 32, 32, 32, 128, 8, 0, 1)),
    ('groupnorm_backward', (24, 32, 32, 32, 128, 8, 1, 1)),
    ('groupnorm_backward', (24, 64, 64, 64, 64, 4, 1, 1)),
    ('groupnorm_backward', (240, 2, 2, 2, 48, 3, 1, 1)),
    ('groupnorm_backward', (240, 2, 2, 2, 72, 4, 0, 1)),
    ('groupnorm_backward', (240, 2, 2, 2, 72, 4, 1, 1)),
    ('groupnorm_backward', (240, 4, 4, 4, 32, 2, 1, 1)),
    ('groupnorm_backward', (240, 4, 4, 4, 48, 3, 0, 1)),
    ('groupnorm_backward', (240, 4, 4, 4, 48, 3, 1, 1)),
    ('groupnorm_backward', (240, 8, 8, 8, 32, 2, 0, 1)),
    ('groupnorm_backward', (240, 8, 8, 8, 32, 2, 1, 1)),
    ('groupnorm_backward', (240, 8, 8, 8, 64, 4, 1, 1)),
    ('groupnorm_backward', (240, 16, 16, 16, 64, 4, 0, 1)),
    ('groupnorm_backward', (240, 16, 16, 16, 64, 4, 1, 1)),
    ('groupnorm_backward', (240, 16, 16, 16, 128, 8, 0, 1)),
    ('groupnorm_backward', (240, 16, 16, 16, 128, 8, 1, 1)),
    ('groupnorm_backward', (240, 32, 32, 32, 32, 2, 1, 1)),
    ('groupnorm_backward', (240, 32, 32, 32, 64, 4, 0, 1)),
    ('groupnorm_backward', (240, 32, 32, 32, 64, 4, 1, 1)),
    ('groupnorm_backward', (240, 64, 64, 64, 32, 2, 1, 1)),
    ('heatmap_head_backward', (24, 16, 16, 16, 256, 24, 0, 1, 10)),
    ('heatmap_head_backward', (240, 16, 16, 16, 128, 24, 1, 0, 10)),
    ('upsample2x', (240, 16, 16, 16, 128)),
    ('upsample2x', (240, 32, 32, 32, 64)),
    ('upsample2x_backward', (240, 32, 32, 32, 128)),
    ('upsample2x_backward', (240, 64, 64, 64, 64)),
]


# --------------------------------------------------------------------------------------------- the method
def owner_map(n, D=ND):
    """Owner of each of n samples: neighbours differ, sample d < D is the first copy of owner d, and every owner has
    copies below sample 64, in [64, 128) and from 128 on (both sides of the 2^31-byte / 2^31-element boundaries of the
    64-channel 64^3 tensors)."""
    own = torch.tensor([(b + b // D) % D for b in range(n)])
    assert all(int(own[b]) == b for b in range(min(n, D)))
    assert bool((own[1:] != own[:-1]).all())
    if n > 128:
        for part in (own[:64], own[64:128], own[128:]):
            assert set(part.tolist()) == set(range(D))
    return own


def copies(own, D=ND):
    return torch.bincount(own, minlength=D).double()


def assert_copies(y, own, chunk_bytes=1 << 30):
    """Every sample of y is bit-identical to the first copy of its owner (compared on the device, in chunks)."""
    n = y.shape[0]
    bits = y.view({2: torch.int16, 4: torch.int32}[y.element_size()])
    rep = own.to(y.device)
    step = max(1, chunk_bytes // (y[0].numel() * y.element_size()))
    for s in range(0, n, step):
        e = min(n, s + step)
        same = (bits[s:e] == bits[rep[s:e]]).reshape(e - s, -1).all(dim=1)
        if not bool(same.all()):
            bad = s + int((~same).nonzero()[0])
            raise AssertionError(f"sample {bad} (copy of {int(own[bad])}) differs from its first copy")


def ncdhw(t, dev="cpu"):
    """act (n, D, H, W, C) -> float64 (n, C, D, H, W)."""
    return t.permute(0, 4, 1, 2, 3).to(dev, torch.float64)


def rel_err(got, ref):
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def report(what, err, bound):
    print(f"  {what}: {err:.3e} (bound {bound:.1e})")
    assert err <= bound, f"{what}: {err:.3e} > {bound:.1e}"


def act_grad_check(what, got, ref, frac_bound, mean_bound):
    """Activation gradient through LeakyReLU(GroupNorm(x)): an element whose pre-activation sits within rounding of 0
    may take the other branch (its gradient then differs by O(1)), so at most `frac_bound` of the elements may differ
    by more than 3e-3 of the largest entry and the mean error is bounded (as in test_groupnorm_backward)."""
    got, ref = got.double().cpu(), ref.double().cpu()
    top = float(ref.abs().max())
    diff = (got - ref).abs()
    frac = float((diff > 3e-3 * top).double().mean())
    mean = float(diff.mean()) / top
    print(f"  {what}: {frac:.2e} of the elements off by > 3e-3 (bound {frac_bound:.0e}), mean error {mean:.3e} "
          f"(bound {mean_bound:.1e}), max {float(diff.max()) / top:.3e}")
    assert frac <= frac_bound and mean <= mean_bound, what


def cuda_gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def randn_act(gen, *shape, scale=1.0):
    return (torch.randn(*shape, generator=gen, device="cuda") * scale).half()


def shapes_of(name):
    return [s for n, s in STEP_SHAPES if n == name]


def _ref_dev(grid):
    """torch's own float64 convolutions: on the device at 64^3 / 32^3 (the CPU takes minutes there), else on the CPU."""
    return "cuda" if grid >= 32 else "cpu"


@pytest.fixture(scope="module")
def ops():
    from neural_marionette_b200 import ops as _ops
    return _ops


@pytest.fixture(autouse=True)
def _free_device_memory():
    yield
    gc.collect()
    if torch.cuda.is_available():
        from neural_marionette_b200 import ops as _ops
        _ops._scratch.clear()                        # grow-only workspaces sized by the full-size launches
        torch.cuda.empty_cache()


@pytest.fixture(scope="module", autouse=True)
def _wall_time():
    t0 = time.perf_counter()
    yield
    print(f"\n[test_gpu_train_scale] wall time {time.perf_counter() - t0:.1f} s")


def test_owner_map_composition_cpu():
    """The method at a tiny size in float64 on the CPU: a batch built with the owner map gives per-sample outputs equal
    to the owner's and batch-reduced outputs equal to sum_d m_d ref_d - for a conv data / weight gradient and for the
    backward of LeakyReLU(GroupNorm(x))."""
    g = torch.Generator().manual_seed(1)
    n, D = 11, ND
    own = owner_map(n, D)
    m = copies(own, D)
    assert float(m.sum()) == n
    x_d = torch.randn(D, 6, 4, 4, 4, generator=g, dtype=torch.float64)
    gy_d = torch.randn(D, 5, 4, 4, 4, generator=g, dtype=torch.float64)
    w = torch.randn(5, 6, 3, 3, 3, generator=g, dtype=torch.float64)
    # conv: data gradient per sample, weight gradient summed over the batch
    dx = torch.nn.grad.conv3d_input((n, 6, 4, 4, 4), w, gy_d[own], padding=1)
    dx_d = torch.nn.grad.conv3d_input((D, 6, 4, 4, 4), w, gy_d, padding=1)
    assert torch.allclose(dx, dx_d[own], rtol=1e-12, atol=1e-12)
    dw = torch.nn.grad.conv3d_weight(x_d[own], w.shape, gy_d[own], padding=1)
    dw_sum = sum(m[d] * torch.nn.grad.conv3d_weight(x_d[d:d + 1], w.shape, gy_d[d:d + 1], padding=1) for d in range(D))
    dw_weighted = torch.nn.grad.conv3d_weight(x_d, w.shape, gy_d * m.view(D, 1, 1, 1, 1), padding=1)
    assert torch.allclose(dw, dw_sum, rtol=1e-12, atol=1e-10) and torch.allclose(dw, dw_weighted, rtol=1e-12, atol=1e-10)
    # GroupNorm (per sample) + LeakyReLU
    gamma = (1 + 0.3 * torch.randn(6, generator=g, dtype=torch.float64)).requires_grad_(True)
    beta = (0.3 * torch.randn(6, generator=g, dtype=torch.float64)).requires_grad_(True)
    dz_d = torch.randn(D, 6, 4, 4, 4, generator=g, dtype=torch.float64)

    def grads(x, dz):
        x = x.clone().requires_grad_(True)
        (F.leaky_relu(F.group_norm(x, 2, gamma, beta, 1e-5), 0.01) * dz).sum().backward()
        out = (x.grad, gamma.grad.clone(), beta.grad.clone())
        gamma.grad = beta.grad = None
        return out
    gx, gg, gb = grads(x_d[own], dz_d[own])
    wx, wg, wb = grads(x_d, dz_d * m.view(D, 1, 1, 1, 1))                 # the composition the GPU tests use
    assert torch.allclose(gx, (wx / m.view(D, 1, 1, 1, 1))[own], rtol=1e-10, atol=1e-12)
    assert torch.allclose(gg, wg, rtol=1e-10, atol=1e-12) and torch.allclose(gb, wb, rtol=1e-10, atol=1e-12)


# --------------------------------------------------------------------------------------------- up-sampling
# fp16 rounding of the output (and, backward, of the two fp16 intermediates between the three axis passes): each at most
# 2^-12 of its value (measured 5.5e-4 / 6.1e-4 backward, 5.8e-4 / 7.0e-4 forward)
UP_BWD_TOL = 1.2e-3
UP_FWD_TOL = 1.5e-3


@gpu
@pytest.mark.parametrize("shape", shapes_of("upsample2x_backward"), ids=str)
def test_upsample2x_backward_full_size(ops, shape):
    """Three-pass trilinear x2 backward: per-sample output, against autograd of F.interpolate."""
    n, D2, H2, W2, C = shape
    own = owner_map(n)
    gy_d = randn_act(cuda_gen(sum(shape)), ND, D2, H2, W2, C)
    got = ops.upsample2x_backward(gy_d[own.cuda()])
    assert got.shape == (n, D2 // 2, H2 // 2, W2 // 2, C)
    assert_copies(got, own)
    first = got[:ND].clone()
    del got
    x = torch.zeros(ND, C, D2 // 2, H2 // 2, W2 // 2, dtype=torch.float64, requires_grad=True)
    F.interpolate(x, scale_factor=2.0, mode="trilinear", align_corners=False).backward(ncdhw(gy_d))
    report(f"upsample2x_backward {shape}", rel_err(ncdhw(first), x.grad), UP_BWD_TOL)


@gpu
@pytest.mark.parametrize("shape", shapes_of("upsample2x"), ids=str)
def test_upsample2x_forward_full_size(ops, shape):
    from neural_marionette_b200 import autograd as AG
    n, D, H, W, C = shape
    own = owner_map(n)
    x_d = randn_act(cuda_gen(7 + sum(shape)), ND, D, H, W, C)
    with torch.no_grad():
        got = AG.Upsample2x.apply(x_d[own.cuda()])
    assert got.shape == (n, 2 * D, 2 * H, 2 * W, C)
    assert_copies(got, own)
    first = got[:ND].clone()
    del got
    ref = F.interpolate(ncdhw(x_d), scale_factor=2.0, mode="trilinear", align_corners=False)
    report(f"upsample2x {shape}", rel_err(ncdhw(first), ref), UP_FWD_TOL)


# --------------------------------------------------------------------------------------------- convolutions
# Data gradients are fp16 tensors: their error is the output rounding, 2^-12 of an entry (measured 2.3e-4 .. 4.7e-4).
DGRAD_TOL = 1e-3
# Weight gradients: fp32 accumulation.  The gather kernels and the k2/s2 / 1x1 layers stay below 3e-5 of the largest
# entry.  The tcgen05 kernel (`conv_wgrad_tc_kernel`, k3 s1 layers with 32-multiple channels) accumulates on the tensor
# cores, whose fp32 accumulator is not rounded to nearest: the error of a CTA's chain grows with its length, ~1e-9 of
# the largest entry per voxel.  The kernel caps a CTA's share at 2048 x 256 voxels (5e-4 .. 7e-4 at most), so the bound
# does not grow with n.
WGRAD_TOL = 1e-4
WGRAD_TC_TOL = 1e-3


def _on_wgrad_tc(D, H, W, Cin, Cout, k, s):
    return k == 3 and s == 1 and Cin % 32 == 0 and Cout % 32 == 0 and Cin <= 256 and Cout <= 256 and W in (16, 32, 64, 128)


@gpu
@pytest.mark.parametrize("key", shapes_of("conv3d_weight_grad"), ids=str)
def test_conv3d_weight_grad_full_size(ops, key):
    """dL/dW summed over the batch (tcgen05 / slab / gather kernel as the step picks it) against sum_d m_d ref_d."""
    n, D, H, W, Cin, Cout, k, s = key
    own = owner_map(n)
    gen = cuda_gen(11 + sum(key))
    x_d = randn_act(gen, ND, D, H, W, Cin)
    gy_d = randn_act(gen, ND, D // s, H // s, W // s, Cout)
    oc = own.cuda()
    got = ops.conv3d_weight_grad(x_d[oc], gy_d[oc], k=k, stride=s)
    dev = _ref_dev(D)
    m = copies(own).to(dev).view(ND, 1, 1, 1, 1)
    ref = torch.nn.grad.conv3d_weight(ncdhw(x_d, dev), (Cout, Cin, k, k, k), ncdhw(gy_d, dev) * m, stride=s,
                                      padding=(k - 1) // 2 if s == 1 else 0)
    report(f"conv3d_weight_grad {key}", rel_err(got, ref), WGRAD_TC_TOL if _on_wgrad_tc(*key[1:]) else WGRAD_TOL)


def _conv(cin, cout, k, s, seed, transposed=False):
    g = torch.Generator().manual_seed(seed)
    conv = (torch.nn.ConvTranspose3d(cin, cout, k, s) if transposed else
            torch.nn.Conv3d(cin, cout, k, s, (k - 1) // 2 if s == 1 else 0))
    with torch.no_grad():
        fan = (cout if transposed else cin) * k ** 3
        conv.weight.copy_((torch.randn(conv.weight.shape, generator=g) / fan ** 0.5).half().float())
        conv.bias.copy_(0.1 * torch.randn(conv.bias.shape, generator=g))
    return conv.cuda()


@gpu
@pytest.mark.parametrize("key", shapes_of("conv3d_input_grad"), ids=str)
def test_conv3d_input_grad_full_size(ops, key):
    """dL/dx of the stride-1 k3 / k1 convs (flipped-tap mirror) and the k2/s2 pool convs (depth-to-space route for
    Cin >= 64, transposed conv otherwise): per-sample output against torch.nn.grad.conv3d_input."""
    n, OD, OH, OW, Cout, Cin, k, s = key
    own = owner_map(n)
    conv = _conv(Cin, Cout, k, s, sum(key))
    gy_d = randn_act(cuda_gen(13 + sum(key)), ND, OD, OH, OW, Cout)
    got = ops.conv3d_input_grad(gy_d[own.cuda()], conv)
    assert got.shape == (n, OD * s, OH * s, OW * s, Cin)
    assert_copies(got, own)
    first = got[:ND].clone()
    del got
    dev = _ref_dev(OD * s)
    ref = torch.nn.grad.conv3d_input((ND, Cin, OD * s, OH * s, OW * s), conv.weight.to(dev, torch.float64),
                                     ncdhw(gy_d, dev), stride=s, padding=conv.padding[0])
    report(f"conv3d_input_grad {key}", rel_err(ncdhw(first), ref), DGRAD_TOL)


@gpu
@pytest.mark.parametrize("key", shapes_of("conv_transpose3d_weight_grad"), ids=str)
def test_conv_transpose3d_weight_grad_full_size(ops, key):
    n, D, H, W, Cin, Cout = key
    own = owner_map(n)
    gen = cuda_gen(17 + sum(key))
    x_d = randn_act(gen, ND, D, H, W, Cin)
    gy_d = randn_act(gen, ND, 2 * D, 2 * H, 2 * W, Cout)
    oc = own.cuda()
    got = ops.conv_transpose3d_weight_grad(x_d[oc], gy_d[oc])
    dev = _ref_dev(2 * D)
    w = torch.zeros(Cin, Cout, 2, 2, 2, dtype=torch.float64, device=dev, requires_grad=True)
    m = copies(own).to(dev).view(ND, 1, 1, 1, 1)
    (F.conv_transpose3d(ncdhw(x_d, dev), w, stride=2) * ncdhw(gy_d, dev) * m).sum().backward()
    report(f"conv_transpose3d_weight_grad {key}", rel_err(got, w.grad), WGRAD_TOL)


@gpu
@pytest.mark.parametrize("key", shapes_of("conv_transpose3d_input_grad"), ids=str)
def test_conv_transpose3d_input_grad_full_size(ops, key):
    n, D2, H2, W2, Cout, Cin = key
    own = owner_map(n)
    conv = _conv(Cin, Cout, 2, 2, sum(key), transposed=True)
    gy_d = randn_act(cuda_gen(19 + sum(key)), ND, D2, H2, W2, Cout)
    got = ops.conv_transpose3d_input_grad(gy_d[own.cuda()], conv)
    assert_copies(got, own)
    dev = _ref_dev(D2)
    ref = F.conv3d(ncdhw(gy_d, dev), conv.weight.to(dev, torch.float64), stride=2)
    report(f"conv_transpose3d_input_grad {key}", rel_err(ncdhw(got[:ND]), ref), DGRAD_TOL)


# --------------------------------------------------------------------------------------------- GroupNorm backward
# fp32 sums over fp16 operands (measured up to 9e-6 of the largest entry), and the fp16 rounding of dL/dx (4.2e-4)
GN_PARAM_TOL = 4e-5
GN_DX_TOL = 1e-3


def _gn(C, groups, seed):
    g = torch.Generator().manual_seed(seed)
    gn = torch.nn.GroupNorm(groups, C)
    with torch.no_grad():
        gn.weight.copy_(1 + 0.3 * torch.randn(C, generator=g))
        gn.bias.copy_(0.3 * torch.randn(C, generator=g))
    return gn


def _gn_normalised(raw_d, gn):
    return F.group_norm(ncdhw(raw_d), gn.num_groups, gn.weight.detach().double().cpu(), gn.bias.detach().double().cpu(),
                        gn.eps)


def _gn_reference(raw_d, dz_d, gn, leaky, m):
    """float64 autograd over LeakyReLU(GroupNorm(raw)) of the distinct samples with dz weighted by the copy counts:
    -> (per-sample dL/draw, sum_d m_d dgamma_d, sum_d m_d dbeta_d, sum_d m_d sum_voxels dL/draw_d)."""
    x = ncdhw(raw_d).requires_grad_(True)
    gamma = gn.weight.detach().double().cpu().requires_grad_(True)
    beta = gn.bias.detach().double().cpu().requires_grad_(True)
    z = F.group_norm(x, gn.num_groups, gamma, beta, gn.eps)
    z = F.leaky_relu(z, 0.01) if leaky else z
    mm = m.view(-1, 1, 1, 1, 1)
    (z * ncdhw(dz_d) * mm).sum().backward()
    return x.grad / mm, gamma.grad, beta.grad, x.grad.sum(dim=(0, 2, 3, 4))


def _gn_producer(n, D, C):
    """(kind, Cin, k, stride) of a layer of the step with output (n, D, D, D, C), a k3 conv where there is one (the
    statistics then come from the tensor-core conv's epilogue, as for most GroupNorms of the step)."""
    convs = sorted(((key[6] != 3, key[4], key[6], key[7]) for key in shapes_of("conv3d_weight_grad")
                    if key[0] == n and key[1] // key[7] == D and key[5] == C))
    if convs:
        return ("conv",) + convs[0][1:]
    convt = [key[4] for key in shapes_of("conv_transpose3d_weight_grad") if key[0] == n and 2 * key[1] == D and key[5] == C]
    if convt:
        return "convT", convt[0], 2, 2
    assert (n, D, D, D, C) in shapes_of("first_conv_weight_grad"), (n, D, C)
    return "first", 4, 5, 1


@gpu
@pytest.mark.parametrize("key", shapes_of("groupnorm_backward"), ids=str)
def test_groupnorm_backward_full_size(ops, key):
    """Backward of [LeakyReLU](GroupNorm(x)) as `ConvGNAct` runs it: with the statistics the producing conv's forward kept
    (`capture_gn_stats`), at every GroupNorm shape of the step; the producer is a layer of the step with that output."""
    n, D, H, W, C, groups, leaky, stats = key
    assert stats, "the step passes the forward's statistics to every GroupNorm backward"
    own = owner_map(n)
    oc = own.cuda()
    gen = cuda_gen(23 + sum(key))
    gn = _gn(C, groups, sum(key))
    gn_c = copy.deepcopy(gn).cuda()
    kind, cin, k, s = _gn_producer(n, D, C)
    conv = _conv(cin, C, k, s, 29 + sum(key), transposed=kind == "convT")
    if kind == "first":                                    # the CoordConv layer reads fractional occupancy
        xin = ((torch.rand(ND, D, H, W, generator=gen, device="cuda") < 0.05).float() *
               torch.randint(1, T + 1, (ND, D, H, W), generator=gen, device="cuda") / T)[oc]
    else:
        din = D // 2 if kind == "convT" else D * s
        xin = randn_act(gen, ND, din, din, din, cin)[oc]
    produce = dict(conv=ops.conv3d, convT=ops.conv_transpose3d, first=ops.first_conv)[kind]
    with ops.capture_gn_stats() as sink:
        raw, _, _ = produce(xin, conv, gn_c)
    del xin
    assert len(sink) == 1 and raw.shape == (n, D, H, W, C)
    st = tuple(sink[0])
    print(f"[groupnorm_backward {key}, statistics from {kind} {cin} -> {C} k{k} s{s}]")
    assert_copies(raw, own)                                            # the forward conv, per sample as well
    dz_d = randn_act(gen, ND, D, H, W, C)
    if leaky:
        # no upstream gradient where the pre-activation sits within rounding of 0: there the kernel's fp32 statistics may
        # pick the other LeakyReLU branch than float64 (a 0.99 * dz difference that the copies multiply by up to 80)
        near0 = _gn_normalised(raw[:ND], gn).abs() < 1e-4
        dz_d = dz_d.masked_fill(near0.permute(0, 2, 3, 4, 1).cuda(), 0.0)
        print(f"  {int(near0.sum())} of {near0.numel()} upstream gradients zeroed (|pre-activation| < 1e-4)")
    dx, dg, db, dxs = ops.groupnorm_backward(raw, dz_d[oc], gn_c, leaky=bool(leaky), stats=st)
    assert_copies(dx, own)
    raw_d, dx_d = raw[:ND].clone(), dx[:ND].clone()
    del raw, dx, st
    m = copies(own)
    rx, rg, rb, rxs = _gn_reference(raw_d, dz_d, gn, bool(leaky), m)
    report("dL/dx", rel_err(ncdhw(dx_d), rx), GN_DX_TOL)
    report("dgamma", rel_err(dg, rg), GN_PARAM_TOL)
    report("dbeta", rel_err(db, rb), GN_PARAM_TOL)
    report("dxsum", rel_err(dxs, rxs), GN_PARAM_TOL)


# --------------------------------------------------------------------------------------------- decoder tail
@gpu
@pytest.mark.parametrize("shape", shapes_of("final_recon_backward_fused"), ids=str)
def test_final_recon_backward_fused_full_size(ops, shape):
    """GN + LeakyReLU + 1x1 conv + tanh / sigmoid + BCE backward of the decoder tail at n = 240, G = 64."""
    n, D, H, W, C = shape
    own = owner_map(n)
    oc = own.cuda()
    gen = torch.Generator().manual_seed(31)
    gn, conv = _gn(C, 2, 37), torch.nn.Conv3d(C, 1, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(1, C, 1, 1, 1, generator=gen) * 0.3)
        conv.bias.fill_(0.1)
    gn_c, conv_c = copy.deepcopy(gn).cuda(), copy.deepcopy(conv).cuda()
    cg = cuda_gen(41)
    raw_d = (torch.randn(ND, D, H, W, C, generator=cg, device="cuda") * 1.3 + 0.2).half()
    ff_d = (torch.rand(ND, D, H, W, generator=cg, device="cuda") < 0.3).float()
    tgt_d = (torch.rand(ND, D, H, W, generator=cg, device="cuda") < 0.3).float()
    gb_d = torch.rand(ND, generator=gen) + 0.5
    raw = raw_d[oc]
    with ops.capture_gn_stats() as sink:
        a, b = ops.gn_scale_shift(raw, gn_c)
    # one frame per "clip": the first-frame map is a per-sample input like the others
    rec, _ = ops.final_recon(raw, a, b, conv_c, ff_d[oc], 1, 10.0, 0.5, target=tgt_d[oc])
    scale = 2.0 ** 10
    draw, dw, db, dg, dbeta, dxs = ops.final_recon_backward_fused(raw, a, b, conv_c, gn_c, sink[0], 10.0, rec, tgt_d[oc],
                                                                 gb_d[own].cuda(), scale)
    del raw, rec
    assert_copies(draw, own)
    draw_d = draw[:ND].clone()
    del draw
    # float64 reference of the distinct samples, the loss weighted by the copy counts
    m = copies(own)
    x = ncdhw(raw_d).requires_grad_(True)
    gnr, convr = copy.deepcopy(gn).double(), copy.deepcopy(conv).double()
    x14 = convr(F.leaky_relu(gnr(x), 0.01))
    recon = torch.sigmoid(10.0 * (torch.tanh(x14) + ff_d.double().cpu()[:, None] - 0.5))
    bce = F.binary_cross_entropy(recon, tgt_d.double().cpu()[:, None], reduction="none").mean(dim=(1, 2, 3, 4))
    (bce * gb_d.double() * m).sum().backward()
    print(f"[final_recon_backward_fused {shape}]")
    act_grad_check("dL/draw", ncdhw(draw_d) / scale, x.grad / m.view(-1, 1, 1, 1, 1), 1e-5, 3e-5)   # measured 0, 4.7e-6
    for name, got, ref in (("dw14", dw, convr.weight.grad), ("db14", db, convr.bias.grad), ("dgamma", dg, gnr.weight.grad),
                           ("dbeta", dbeta, gnr.bias.grad), ("dxsum", dxs, x.grad.sum(dim=(0, 2, 3, 4)))):
        report(name, rel_err(got, ref), 4e-6)             # fp32 sums over 6.3e7 voxels: measured <= 6.3e-7 (db14)


# --------------------------------------------------------------------------------------------- CoordConv weight gradient
@gpu
@pytest.mark.parametrize("key", shapes_of("first_conv_weight_grad"), ids=str)
def test_first_conv_weight_grad_full_size(ops, key):
    """Per-frame branch (240 binary frames) and clip-mean branch (24 fractional frames, the mean over 10 frames)."""
    n, Gd, _, _, Cout = key
    own = owner_map(n)
    oc = own.cuda()
    cg = cuda_gen(43 + n)
    occ_d = (torch.rand(ND, Gd, Gd, Gd, generator=cg, device="cuda") < 0.05).float()
    if n < B * T:                                          # the spatio-temporal branch sees the clip's frame mean
        occ_d = occ_d * torch.randint(1, T + 1, (ND, Gd, Gd, Gd), generator=cg, device="cuda") / T
    gy_d = randn_act(cg, ND, Gd, Gd, Gd, Cout, scale=Gd ** -1.5)
    got = ops.first_conv_weight_grad(occ_d[oc], gy_d[oc])
    m = copies(own).cuda().view(ND, 1, 1, 1, 1)
    ref = torch.nn.grad.conv3d_weight(O.add_coord_channels(occ_d[:, None].double()), (Cout, 4, 5, 5, 5),
                                      ncdhw(gy_d, "cuda") * m, padding=2)
    print(f"[first_conv_weight_grad {key}]")
    for c in range(4):
        report(f"input channel {c}", rel_err(got[:, c], ref[:, c]), 3e-6)                      # measured <= 6.7e-7


# --------------------------------------------------------------------------------------------- heads, adjust, chamfer
# fp16 activation gradients: output rounding (measured <= 3.9e-4); fp32 parameter gradients (measured <= 6.1e-6)
HEAD_ACT_TOL, HEAD_PARAM_TOL = 1e-3, 3e-5


def _clip_owner(nclips=B):
    own_c = owner_map(nclips)
    return own_c, (own_c[:, None] * T + torch.arange(T)).reshape(-1)      # clip owners; frame -> frame of clip d


def _act_grad_near0_check(what, got, ref, u, top_tol):
    """An activation gradient through LeakyReLU(u) per voxel (channels on dim 1): a voxel may be off only where some
    float64 pre-activation u of it sits within 1e-4 of 0 (fp32 may take the other branch there, an O(1) change of that
    term); everywhere else the error stays within `top_tol` of the largest entry."""
    got, ref = got.detach().double().cpu(), ref.detach().double().cpu()
    top = float(ref.abs().max())
    err = ((got - ref).abs().amax(dim=1) / top)
    near = (u.detach().abs() < 1e-4).any(dim=1)
    far = float(err[~near].max())
    print(f"  {what}: {far:.3e} (bound {top_tol:.1e}) off the voxels with a pre-activation within 1e-4 of 0 "
          f"({int(near.sum())} of {near.numel()}; worst there {float(err[near].max()) if near.any() else 0.0:.3e})")
    assert far <= top_tol, what


@gpu
@pytest.mark.parametrize("k", [K, 64])
def test_heatmap_head_backward_full_size(ops, k):
    """Both heads, the propagate conv, Softplus, soft-argmax and the heat-map mean at g = 16, B = 24, T = 10 (clips as
    the distinct unit: the spatio-temporal head couples a clip's frames)."""
    from neural_marionette_b200 import autograd as AG
    g = G // 4
    own_c, own_f = _clip_owner()
    gen = torch.Generator().manual_seed(47 + k)
    feat = torch.randn(ND * T, 128, g, g, g, generator=gen).half().double()
    fst = torch.randn(ND, 256, g, g, g, generator=gen).half().double()
    head, hst, prop = torch.nn.Conv3d(128, k, 1), torch.nn.Conv3d(256, k, 1), torch.nn.Conv3d(2, 1, 1)
    with torch.no_grad():
        head.weight.copy_(torch.randn(head.weight.shape, generator=gen) / 128 ** 0.5)
        head.bias.copy_(0.1 * torch.randn(k, generator=gen))
        hst.weight.copy_(torch.randn(hst.weight.shape, generator=gen) / 256 ** 0.5)
        hst.bias.copy_(0.1 * torch.randn(k, generator=gen))
        prop.weight.copy_(torch.tensor([0.9, 0.6]).view(1, 2, 1, 1, 1))
        prop.bias.fill_(-0.3)
    dkp = torch.randn(ND * T, k, 4, generator=gen)
    dhm = torch.randn(ND * T, k, generator=gen)
    # float64 reference of the distinct clips, the upstream gradients weighted by the copy counts
    m = copies(own_c)
    mf = m.repeat_interleave(T)
    head_r, hst_r, prop_r = (copy.deepcopy(x).double() for x in (head, hst, prop))
    feat_r, fst_r = feat.clone().requires_grad_(True), fst.clone().requires_grad_(True)
    u_st = hst_r(fst_r)
    u = head_r(feat_r)
    prev = F.leaky_relu(u_st, 0.01)
    pv = prev.repeat_interleave(T, 0).reshape(ND * T * k, 1, g, g, g)
    hm = F.softplus(prop_r(torch.cat([F.leaky_relu(u, 0.01).view(ND * T * k, 1, g, g, g), pv], 1))).view(ND * T, k, g, g, g)
    kp = O.keypoints_from_heatmap(hm)
    top2 = hm.detach().mean(dim=(2, 3, 4)).topk(2, dim=1).values
    assert float(((top2[:, 0] - top2[:, 1]) / top2[:, 0]).min()) > 1e-5      # the intensity's argmax is not a near tie
    ((kp * dkp.double() * mf.view(-1, 1, 1)).sum() + (hm.mean(dim=(2, 3, 4)) * dhm.double() * mf.view(-1, 1)).sum()).backward()
    # the kernels through the autograd Functions on the full batch
    head_c, hst_c, prop_c = (copy.deepcopy(x).cuda() for x in (head, hst, prop))
    ops.set_grad_scale(256.0)
    fa = feat.float().permute(0, 2, 3, 4, 1).contiguous().half().cuda()[own_f.cuda()].requires_grad_(True)
    fs = fst.float().permute(0, 2, 3, 4, 1).contiguous().half().cuda()[own_c.cuda()].requires_grad_(True)
    link = {}
    prev_c = AG.HeadST.apply(fs, hst_c.weight, hst_c.bias, hst_c, k, link)
    heat_c, kp_c, mean_c = AG.Head.apply(fa, head_c.weight, head_c.bias, prev_c, prop_c.weight, prop_c.bias, head_c, prop_c,
                                         k, T, 1.5, link)
    ((kp_c * dkp.cuda()[own_f.cuda()]).sum() + (mean_c * dhm.cuda()[own_f.cuda()]).sum()).backward()
    for t in (kp_c.detach(), fa.grad, fs.grad):
        assert_copies(t.reshape(B, -1), own_c)
    print(f"[heatmap head backward, K = {k}]")
    report("keypoints (forward)", float((kp_c.detach()[:ND * T].cpu() - kp.detach()).abs().max()), 2e-6)
    _act_grad_near0_check("d feature", ncdhw(fa.grad[:ND * T]) / 256.0, feat_r.grad / mf.view(-1, 1, 1, 1, 1), u,
                          HEAD_ACT_TOL)
    _act_grad_near0_check("d st feature", ncdhw(fs.grad[:ND]) / 256.0, fst_r.grad / m.view(-1, 1, 1, 1, 1), u_st,
                          HEAD_ACT_TOL)
    for name, a, r in (("head w", head_c.weight, head_r.weight), ("head b", head_c.bias, head_r.bias),
                       ("st w", hst_c.weight, hst_r.weight), ("st b", hst_c.bias, hst_r.bias),
                       ("prop w", prop_c.weight, prop_r.weight), ("prop b", prop_c.bias, prop_r.bias)):
        report(name, rel_err(a.grad, r.grad), HEAD_PARAM_TOL)


@gpu
@pytest.mark.parametrize("k", [K, 64])
def test_decoder_adjust_backward_full_size(ops, k):
    """Gaussian render + adjust conv at g = 16, B = 24, T = 10: d first_feature (per clip), d keypoints (per frame),
    dW, db (batch sums)."""
    from neural_marionette_b200 import autograd as AG
    g = G // 4
    own_c, own_f = _clip_owner()
    gen = torch.Generator().manual_seed(53 + k)
    ff = torch.randn(ND, 128, g, g, g, generator=gen).half().double()
    kp = torch.cat([torch.rand(ND * T, k, 3, generator=gen) * 1.4 - 0.7, torch.rand(ND * T, k, 1, generator=gen) * 0.8 + 0.2], -1)
    conv = torch.nn.Conv3d(128 + 2 * k + 3, 128, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=gen) / conv.in_channels ** 0.5)
        conv.bias.copy_((torch.rand(128, generator=gen) * 2 - 1) / conv.in_channels ** 0.5)
    gy = torch.randn(ND * T, 128, g, g, g, generator=gen).half().double()
    conv_c = copy.deepcopy(conv).cuda()
    ops.set_grad_scale(64.0)
    ffa = ff.float().permute(0, 2, 3, 4, 1).contiguous().half().cuda()[own_c.cuda()].requires_grad_(True)
    kpc = kp.cuda()[own_f.cuda()].requires_grad_(True)
    yc = AG.Adjust.apply(ffa, kpc, conv_c.weight, conv_c.bias, conv_c, T, g, k, 1.5)
    yc.backward((gy.float().permute(0, 2, 3, 4, 1).contiguous().cuda()[own_f.cuda()] * 64.0).half())
    for t in (yc.detach(), ffa.grad, kpc.grad):
        assert_copies(t.reshape(B, -1), own_c)
    # float64 reference.  The LeakyReLU branch of every element is borrowed on purpose from the kernel's own fp16 forward
    # output (checked against float64 below), so that elements within rounding of 0 do not enter as O(1) differences.
    m = copies(own_c)
    mf = m.repeat_interleave(T)
    conv_r = copy.deepcopy(conv).double()
    ff_r, kp_r = ff.clone().requires_grad_(True), kp.double().clone().requires_grad_(True)
    gs = O.render_gaussians(kp_r, 1.5, g).view(ND, T, k, g, g, g)
    pre = torch.stack([conv_r(O.add_coord_channels(torch.cat([gs[:, t], ff_r, gs[:, 0]], 1))) for t in range(T)], 1)
    pre = pre.reshape(ND * T, 128, g, g, g)
    y_first = ncdhw(yc.detach()[:ND * T])
    y = pre * torch.where(y_first > 0, 1.0, 0.01)
    (y * gy * mf.view(-1, 1, 1, 1, 1)).sum().backward()
    print(f"[decoder adjust backward, K = {k}]")
    report("forward", rel_err(y_first, y.detach()), 1.5e-3)                                     # measured 4.3e-4
    report("d first feature", rel_err(ncdhw(ffa.grad[:ND]) / 64.0, ff_r.grad / m.view(-1, 1, 1, 1, 1)), HEAD_ACT_TOL)
    report("d keypoints", rel_err(kpc.grad[:ND * T], kp_r.grad / mf.view(-1, 1, 1)), 4e-6)       # measured <= 9.5e-7
    report("dW", rel_err(conv_c.weight.grad, conv_r.weight.grad), 4e-6)
    report("db", rel_err(conv_c.bias.grad, conv_r.bias.grad), 4e-6)


@gpu
@pytest.mark.parametrize("k", [K, 64])
def test_chamfer_backward_full_size(ops, k):
    """Chamfer volume-fitting loss backward at G = 64 over 240 frames (per-frame output)."""
    own = owner_map(B * T)
    gen = torch.Generator().manual_seed(59 + k)
    seq = (torch.rand(ND, G, G, G, generator=gen) < 0.08).float()
    kp = torch.cat([torch.rand(ND, k, 3, generator=gen) * 1.6 - 0.8, torch.rand(ND, k, 1, generator=gen)], -1)
    go = torch.rand(ND, generator=gen) + 0.5
    oc = own.cuda()
    got = ops.chamfer_vol_fit_backward(seq.cuda()[oc], kp.cuda()[oc], go.cuda()[oc])
    assert_copies(got, own)
    kp_r = kp.double().requires_grad_(True)
    (O.chamfer_vol_fit(seq.double().view(1, ND, 1, G, G, G), kp_r.view(1, ND, k, 4)) * go.double()).sum().backward()
    report(f"chamfer backward K = {k}", rel_err(got[:ND], kp_r.grad), 2e-6)                  # measured <= 4.9e-7


# --------------------------------------------------------------------------------------------- the assembled step
def _net(seed=0):
    import neural_marionette_b200 as nm
    hp = O.default_hparams(grid_size=G, Tcond=3, Ttot=10)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(O.synthetic_state_dict(hp, seed=seed), strict=True)
    net = net.cuda().train()
    net.anneal(1)
    return net


_RECORDED = ("upsample2x", "upsample2x_backward", "conv3d_input_grad", "conv3d_weight_grad", "conv_transpose3d_weight_grad",
             "conv_transpose3d_input_grad", "groupnorm_backward", "final_recon_backward_fused", "final_recon_backward",
             "first_conv_weight_grad", "heatmap_head_backward", "decoder_adjust_backward", "chamfer_vol_fit_backward")


def _shape_key(name, args, kw):
    """What of a call picks the kernel and its tiling: tensor shapes, channel counts, kernel sizes, modes."""
    a0 = tuple(args[0].shape)
    if name in ("upsample2x", "upsample2x_backward", "final_recon_backward_fused", "final_recon_backward"):
        return a0
    if name == "conv3d_input_grad":                         # (n, OD, OH, OW, Cout, Cin, k, stride)
        conv = args[1]
        return a0 + (conv.in_channels, conv.kernel_size[0], conv.stride[0])
    if name == "conv3d_weight_grad":                        # (n, D, H, W, Cin, Cout, k, stride)
        return a0 + (args[1].shape[-1], kw.get("k", 3), kw.get("stride", 1))
    if name == "conv_transpose3d_weight_grad":              # (n, D, H, W, Cin, Cout)
        return a0 + (args[1].shape[-1],)
    if name == "conv_transpose3d_input_grad":               # (n, 2D, 2H, 2W, Cout, Cin)
        return a0 + (args[1].in_channels,)
    if name == "groupnorm_backward":                        # (n, D, H, W, C, groups, leaky, forward statistics)
        return a0 + (args[2].num_groups, int(kw.get("leaky", True)), int(kw.get("stats") is not None))
    if name == "first_conv_weight_grad":                    # (n, G, G, G, Cout)
        return a0 + (args[1].shape[-1],)
    if name == "heatmap_head_backward":                     # (n, g, g, g, C, K, mode, summed over frames, T)
        return a0 + (args[2], args[3], int(kw.get("dq_in") is not None), kw.get("frames_per_clip", 1))
    if name == "decoder_adjust_backward":                   # (B, g, g, g, 128, T, g, K)
        return tuple(args[2].shape) + tuple(args[5:8])
    if name == "chamfer_vol_fit_backward":                  # (n, G, G, G, K)
        return a0 + (args[1].shape[1],)
    raise KeyError(name)


def record_step_shapes(nclips=B, frames=T, seed=0):
    """One training step (forward + backward of the stage-1 loss sum) with every backward entry point of `ops` wrapped:
    -> sorted distinct (entry point, shape key)."""
    from neural_marionette_b200 import ops
    seen = set()
    saved = {name: getattr(ops, name) for name in _RECORDED}

    def wrap(name, fn):
        def inner(*args, **kw):
            seen.add((name, _shape_key(name, args, kw)))
            return fn(*args, **kw)
        return inner
    net = _net(seed)
    raw = torch.from_numpy(np.stack([O.synthetic_clip(4000 + b, frames, 5000) for b in range(nclips)], 0)).cuda()
    try:
        for name in _RECORDED:
            setattr(ops, name, wrap(name, saved[name]))
        vox = ops.normalize_voxelize(raw, G, check=False)
        OG.detector_loss(net.kypt_detector(vox), recon_only=False).backward()
        torch.cuda.synchronize()
    finally:
        for name in _RECORDED:
            setattr(ops, name, saved[name])
    return sorted(seen)


@gpu
def test_step_shapes_are_all_listed():
    """Every (backward entry point, shape) of a real 24 x 10 step at G = 64 is in STEP_SHAPES, so the full-size tests
    above cover it; a change that makes the step launch a new shape fails here."""
    got = record_step_shapes()
    missing = [s for s in got if s not in set(STEP_SHAPES)]
    assert not missing, f"shapes the step runs that STEP_SHAPES does not list: {missing}"


# measured: whole-gradient error 2.3e-4, lowest cosine 0.999995, loss 7.7e-8 relative
STEP_WHOLE_TOL, STEP_COS_TOL, STEP_LOSS_TOL = 1e-3, 0.99998, 1e-6


@gpu
def test_full_size_step_is_the_sum_of_its_clips():
    """The 24 x 10 step at G = 64 on a batch of D distinct clips against the same CUDA step on each clip alone: GroupNorm
    is per sample and every loss term is a mean over clips, so grad = sum_d (m_d / 24) g_d up to loss-scale rounding and
    summation order; the forward outputs of every copy of a clip are bit-identical."""
    own = owner_map(B)
    m = copies(own)
    vox_d = torch.from_numpy(np.stack([O.voxelize_clip(O.episodic_normalization(O.synthetic_clip(5100 + d, T, 5000)), G)
                                       for d in range(ND)], 0)).float().cuda()
    net = _net(3)
    det = net.kypt_detector
    params = [(k, p) for k, p in det.named_parameters() if p.requires_grad]

    def step(vox):
        for _, p in params:
            p.grad = None
        out = det(vox)
        loss = OG.detector_loss(out, recon_only=False)
        loss.backward()
        return out, loss.detach(), {k: p.grad.detach().double().clone() for k, p in params if p.grad is not None}
    out, loss, grads = step(vox_d[own.cuda()].contiguous())
    for key in ("keypoints", "heatmaps", "recon", "first_feature"):
        assert_copies(out[key].detach(), own)
    del out
    torch.cuda.empty_cache()
    ref, ref_loss = {}, 0.0
    for d in range(ND):
        _, loss_d, g_d = step(vox_d[d:d + 1].contiguous())
        ref_loss += float(m[d]) / B * float(loss_d)
        for k, v in g_d.items():
            ref[k] = ref.get(k, 0.0) + float(m[d]) / B * v
    assert sorted(ref) == sorted(grads)
    allg = torch.cat([grads[k].reshape(-1) for k in sorted(grads)])
    allr = torch.cat([ref[k].reshape(-1) for k in sorted(grads)])
    whole = float((allg - allr).norm() / allr.norm())
    cos = {k: float((grads[k] * ref[k]).sum() / (grads[k].norm() * ref[k].norm()).clamp_min(1e-300)) for k in grads
           if float(ref[k].norm()) > 0}
    worst = min(cos, key=cos.get)
    print(f"[full-size step] loss {float(loss):.6f} vs sum of clips {ref_loss:.6f}; whole-gradient relative L2 error "
          f"{whole:.3e} (bound {STEP_WHOLE_TOL:.0e}); lowest per-tensor cosine {cos[worst]:.6f} ({worst}, bound "
          f"{STEP_COS_TOL})")
    assert abs(float(loss) - ref_loss) <= STEP_LOSS_TOL * abs(ref_loss)
    assert whole <= STEP_WHOLE_TOL
    assert cos[worst] >= STEP_COS_TOL


if __name__ == "__main__":                                     # PYTHONPATH=. python tests/test_gpu_train_scale.py
    torch.cuda.reset_peak_memory_stats()
    t0 = time.perf_counter()
    shapes = record_step_shapes()
    print(f"# one {B} x {T} step at G = {G}: {time.perf_counter() - t0:.1f} s, peak "
          f"{torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB allocated")
    print("STEP_SHAPES = [")
    for s in shapes:
        print(f"    {s!r},")
    print("]")
