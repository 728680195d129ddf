"""GPU parity tests, kernel by kernel, through the C ABI (ops.* are 1:1 wrappers of include/nm_b200.h).
The checker is the CPU oracle (oracle/nm_oracle.py, pinned to the reference by tests/golden/).

Tolerances (BASELINE.json north_star): occupancy grids bit-exact; keypoints <= 1e-3 of the grid extent
(extent = 2 -> 2e-3 absolute); heat-maps <= 1e-2 relative to the tensor's peak.  Per-kernel tests are much
tighter: fp16 activations carry 2^-11 relative rounding, accumulation is fp32.
"""
import hashlib
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import nm_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from neural_marionette_b200 import ops as _ops
    return _ops


def to_act(x):  # NCDHW fp32 cpu -> channels-last fp16 cuda
    return x.permute(0, 2, 3, 4, 1).contiguous().half().cuda()


def from_act(y):  # channels-last fp16 cuda -> NCDHW fp32 cpu
    return y.float().cpu().permute(0, 4, 1, 2, 3).contiguous()


def rel_err(got, ref):
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-6))


# ------------------------------------------------------------------------------------------------ voxelize
def test_voxelize_bit_exact_golden(golden_dir):
    import neural_marionette_b200 as nm
    cases = json.load(open(os.path.join(golden_dir, "voxelize_hashes.json")))
    done = set()
    for c in cases:
        key = (c["seed"], c["N"], c["G"])
        if key in done:
            continue
        done.add(key)
        T = 1 + max(x["t"] for x in cases if x["seed"] == c["seed"])
        raw = O.synthetic_clip(c["seed"], T, c["N"])
        pts = O.episodic_normalization(raw)                              # float64, as the reference produces
        grid = nm.voxelize_clip(pts, c["G"]).cpu().numpy()               # (T, 1, G, G, G)
        fused = nm.voxelize_raw_clips(raw[None], c["G"])[0].cpu().numpy()
        for x in (x for x in cases if x["seed"] == c["seed"]):
            g = grid[x["t"]]
            assert g.dtype == np.float32 and int(g.sum()) == x["occupied"]
            assert hashlib.sha256(np.ascontiguousarray(g).tobytes()).hexdigest() == x["sha256"]
            assert np.array_equal(fused[x["t"]], g), "fused normalise+voxelize differs"


def test_voxelize_numpy_dropin_and_real_geometry(golden_dir):
    import neural_marionette_b200 as nm
    z = np.load(os.path.join(golden_dir, "voxelize_obj.npz"))
    pts = O.episodic_normalization(z["obj_points_f32"][None], 0.8)[0]
    g = nm.voxelize(pts, (64, 64, 64), is_binarized=True)
    assert g.shape == (1, 64, 64, 64) and g.dtype == np.float32
    assert np.array_equal(np.packbits(g.astype(np.uint8).ravel()), z["obj_grid_packed"])
    fused = nm.voxelize_raw_clips(z["obj_points_f32"][None, None], 64, scale=0.8)[0, 0].cpu().numpy()
    assert np.array_equal(fused, g)


def test_voxelize_edge_cases():
    import neural_marionette_b200 as nm
    assert nm.voxelize(np.zeros((0, 3)), (8, 8, 8)).sum() == 0                      # empty cloud
    p = np.array([[0.0, 0.0, 0.0]] * 70 + [[np.nextafter(1.0, 0.0)] * 3, [-1.0, -1.0, -1.0]])
    g = nm.voxelize(p, (8, 8, 8))
    assert np.array_equal(g, O.voxelize(p, (8, 8, 8)))                              # duplicates, both extremes
    assert np.array_equal(nm.voxelize(p.astype(np.float32), (16,) * 3), O.voxelize(p.astype(np.float32), (16,) * 3))
    with pytest.raises(ValueError):                                                 # numpy would raise IndexError
        nm.voxelize(np.array([[1.5, 0.0, 0.0]]), (8, 8, 8))
    rng = np.random.default_rng(0)                                                  # ragged sizes, heavy collisions
    for n in (1, 31, 33, 255, 257, 100000):
        q = rng.uniform(-1, 1, size=(n, 3)) * 0.2
        assert np.array_equal(nm.voxelize(q, (128,) * 3), O.voxelize(q, (128,) * 3))


def test_voxelize_translation_variants():
    import neural_marionette_b200 as nm
    raw = O.synthetic_clip(1004, 2, 5000)
    for scale, xt, zt in [(0.8, 0.0, 0.0), (0.7, 0.1, 0.05)]:
        ref = O.voxelize_clip(O.episodic_normalization(raw, scale, xt, zt), 64)
        got = nm.voxelize_raw_clips(raw[None], 64, scale, xt, zt)[0].cpu().numpy()
        assert np.array_equal(got, ref)


# ------------------------------------------------------------------------------------------------ convolutions
CONV_CASES = [
    # (n, grid, Cin, Cout, k, stride)
    (2, 8, 64, 64, 1, 1), (2, 8, 64, 64, 3, 1), (1, 16, 32, 64, 3, 1), (1, 16, 64, 32, 3, 1),
    (1, 16, 128, 64, 3, 1), (1, 8, 128, 256, 3, 1), (1, 8, 256, 256, 1, 1), (3, 4, 48, 48, 3, 1),
    (5, 2, 72, 72, 3, 1), (20, 2, 48, 72, 3, 1), (2, 16, 32, 32, 2, 2), (2, 8, 64, 64, 2, 2),
    (3, 4, 48, 48, 2, 2), (1, 32, 32, 32, 3, 1), (2, 8, 32, 64, 1, 1), (3, 2, 48, 48, 2, 2),
    (2, 16, 32, 48, 3, 1), (1, 16, 64, 16, 3, 1),   # k3 at 16^3, Cout not a multiple of 32: conv3d_tc_kernel
]


@pytest.mark.parametrize("n,grid,cin,cout,k,stride", CONV_CASES)
def test_conv3d_tc(ops, n, grid, cin, cout, k, stride):
    g = torch.Generator().manual_seed(n * 1000 + grid * 10 + cin + cout + k)
    conv = torch.nn.Conv3d(cin, cout, k, stride, (k - 1) // 2 if stride == 1 else 0)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * k ** 3) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g))
    x = torch.randn(n, cin, grid, grid, grid, generator=g)
    xh = x.half().float()
    wh = conv.weight.detach().half().float()
    ref = F.conv3d(xh, wh, conv.bias.detach(), stride=stride, padding=conv.padding)
    conv = conv.cuda()
    got = from_act(ops.conv3d(to_act(x), conv))
    chk = from_act(ops.conv3d_direct(to_act(x), conv))
    torch.cuda.synchronize()
    assert rel_err(chk, F.conv3d(xh, conv.weight.detach().cpu(), conv.bias.detach().cpu(), stride=stride,
                                 padding=conv.padding)) < 3e-3, "direct (CUDA-core) conv wrong"
    err = rel_err(got, ref)
    if err >= 2e-3:  # leave evidence for offline diagnosis
        os.makedirs("gpurun_out", exist_ok=True)
        np.savez_compressed(f"gpurun_out/conv_fail_{n}_{grid}_{cin}_{cout}_{k}_{stride}.npz", got=got.numpy(),
                            ref=ref.numpy(), x=xh.numpy(), w=wh.numpy())
    assert err < 2e-3, f"tcgen05 conv rel err {err}"
    # GroupNorm statistics fused into the conv epilogue == statistics of the stored output
    if cout % 16 == 0:
        gn = torch.nn.GroupNorm(cout // 16, cout).cuda()
        with torch.no_grad():
            gn.weight.copy_(1 + 0.3 * torch.randn(cout, generator=g))
            gn.bias.copy_(0.3 * torch.randn(cout, generator=g))
        raw, a, b = ops.conv3d(to_act(x), conv, gn)
        a2, b2 = ops.gn_scale_shift(raw, gn)
        assert torch.equal(raw, ops.conv3d(to_act(x), conv))
        assert (a - a2).abs().max() <= 2e-3 * a2.abs().max() and (b - b2).abs().max() <= 2e-3 * (1 + b2.abs().max())


@pytest.mark.parametrize("n,grid,cin,cout", [(2, 16, 64, 64), (1, 32, 64, 32), (3, 16, 64, 64), (2, 16, 32, 32),
                                             (1, 32, 32, 32)])
def test_conv3d_fused_input_groupnorm(ops, n, grid, cin, cout):
    """conv(LeakyReLU(GroupNorm(raw))) with the normalisation applied inside the conv's operand path."""
    g = torch.Generator().manual_seed(cin * 7 + cout)
    conv = torch.nn.Conv3d(cin, cout, 3, 1, 1).cuda()
    gn_out = torch.nn.GroupNorm(cout // 16, cout).cuda()
    raw_in = to_act(torch.randn(n, cin, grid, grid, grid, generator=g) * 1.5 + 0.3)
    a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
    b = torch.randn(n, cin, generator=g).cuda()
    assert ops.can_fuse_input(raw_in, conv)
    assert not ops.can_fuse_input(to_act(torch.zeros(1, 128, 16, 16, 16)), torch.nn.Conv3d(128, 64, 3, 1, 1).cuda())
    ref_in = ops.affine_act(raw_in, a, b, True)                       # separate pass (rounds to fp16)
    ref, ra, rb = ops.conv3d(ref_in, conv, gn_out)
    got, ga, gb = ops.conv3d(raw_in, conv, gn_out, in_affine=(a, b, True))
    torch.cuda.synchronize()
    assert rel_err(got.float().cpu(), ref.float().cpu()) < 2e-3      # same arithmetic up to fp16 rounding order
    assert (ga - ra).abs().max() <= 2e-3 * ra.abs().max() and (gb - rb).abs().max() <= 2e-3 * (1 + rb.abs().max())
    # borders: the zero padding must stay zero AFTER the affine (shift != 0)
    x = torch.zeros(1, cin, grid, grid, grid)
    x[:, :, 0, 0, 0] = 1.0
    a1, b1 = torch.ones(1, cin).cuda(), torch.full((1, cin), 0.7).cuda()
    got = ops.conv3d(to_act(x), conv, in_affine=(a1, b1, False))
    ref = ops.conv3d(ops.affine_act(to_act(x), a1, b1, False), conv)
    assert rel_err(got.float().cpu(), ref.float().cpu()) < 2e-3


@pytest.mark.parametrize("n,grid,cin,cout,fused", [(2, 16, 64, 32, True), (1, 32, 64, 32, False), (3, 16, 64, 64, True),
                                                   (1, 32, 64, 64, True), (2, 16, 128, 64, False), (1, 32, 128, 64, False)])
def test_conv3d_upsample_fused(ops, n, grid, cin, cout, fused):
    """conv3d_k3(upsample2x(LeakyReLU(GN(raw)))) with the up-sampled tensor interpolated inside the conv's operand
    path: against the two-kernel device path and against torch (F.interpolate trilinear + conv3d)."""
    g = torch.Generator().manual_seed(grid + cout + cin)
    conv = torch.nn.Conv3d(cin, cout, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * 27) ** 0.5)
    gn_out = torch.nn.GroupNorm(cout // 16, cout).cuda()
    lo = grid // 2
    x = torch.randn(n, cin, lo, lo, lo, generator=g) * 1.5 + 0.3
    raw = to_act(x)
    a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
    b = torch.randn(n, cin, generator=g).cuda()
    conv = conv.cuda()
    assert ops.can_conv_up2x(raw, conv)
    if fused:
        act = ops.affine_act(raw, a, b, True)
        got, ga, gb = ops.conv3d_up2x(raw, conv, gn_out, in_affine=(a, b, True))
    else:
        act = raw
        got, ga, gb = ops.conv3d_up2x(raw, conv, gn_out)
    two, ta, tb = ops.conv3d(ops.upsample2x(act), conv, gn_out)
    ref = F.conv3d(F.interpolate(from_act(act), scale_factor=2.0, mode="trilinear", align_corners=False),
                   conv.weight.detach().cpu().half().float(), conv.bias.detach().cpu(), padding=1)
    torch.cuda.synchronize()
    assert rel_err(from_act(two), ref) < 3e-3
    assert rel_err(from_act(got), ref) < 3e-3
    assert rel_err(from_act(got), from_act(two)) < 3e-3
    assert (ga - ta).abs().max() <= 3e-3 * ta.abs().max() and (gb - tb).abs().max() <= 3e-3 * (1 + tb.abs().max())


@pytest.mark.parametrize("n,grid,cin,cout,k,stride", [(2, 16, 32, 32, 2, 2), (1, 32, 32, 32, 2, 2), (3, 8, 32, 64, 1, 1),
                                                     (2, 16, 32, 64, 1, 1), (5, 16, 32, 32, 1, 1), (2, 16, 64, 64, 2, 2),
                                                     (1, 32, 64, 64, 2, 2), (3, 16, 64, 128, 1, 1), (2, 8, 64, 64, 1, 1)])
def test_conv3d_pointwise_fused_input(ops, n, grid, cin, cout, k, stride):
    """Cin = 32 / 64 pool / 1x1 convs on the memory-pipe kernel: plain, with the producer's GroupNorm + LeakyReLU
    applied in registers, and (64->64 pool) with the two normalised branches of a Res3DBlock summed on the fly;
    GroupNorm statistics of the output from the accumulators."""
    g = torch.Generator().manual_seed(grid * 3 + cin + cout + k)
    conv = torch.nn.Conv3d(cin, cout, k, stride, 0)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * k ** 3) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g))
    gn_out = torch.nn.GroupNorm(cout // 16, cout).cuda()
    x = torch.randn(n, cin, grid, grid, grid, generator=g) * 1.5 + 0.3
    raw_in = to_act(x)
    assert ops._pw_ok(raw_in, conv) and ops.can_fuse_input(raw_in, conv)
    wh, bias = conv.weight.detach().half().float(), conv.bias.detach().clone()
    ref = F.conv3d(x.half().float(), wh, bias, stride=stride)
    conv = conv.cuda()
    assert rel_err(from_act(ops.conv3d(raw_in, conv)), ref) < 2e-3
    a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
    b = torch.randn(n, cin, generator=g).cuda()
    bc = lambda v: v.cpu()[:, :, None, None, None]                        # noqa: E731
    lin_in = x.half().float() * bc(a) + bc(b)
    ref2 = F.conv3d(F.leaky_relu(lin_in, 0.01).half().float(), wh, bias, stride=stride)
    got, ga, gb = ops.conv3d(raw_in, conv, gn_out, in_affine=(a, b, True))
    torch.cuda.synchronize()
    assert rel_err(from_act(got), ref2) < 2e-3
    ra, rb = ops.gn_scale_shift(got, gn_out)
    assert (ga - ra).abs().max() <= 2e-3 * ra.abs().max() and (gb - rb).abs().max() <= 2e-3 * (1 + rb.abs().max())
    # no activation: pure affine
    got3 = ops.conv3d(raw_in, conv, in_affine=(a, b, False))
    assert rel_err(from_act(got3), F.conv3d(lin_in.half().float(), wh, bias, stride=stride)) < 2e-3
    if ops.can_fuse_input2(raw_in, conv):
        x2 = torch.randn(n, cin, grid, grid, grid, generator=g)
        a2 = (0.5 + torch.rand(n, cin, generator=g)).cuda()
        b2 = torch.randn(n, cin, generator=g).cuda()
        for a2_, b2_ in ((a2, b2), (None, None)):
            second = x2.half().float() * bc(a2_) + bc(b2_) if a2_ is not None else x2.half().float()
            ref4 = F.conv3d((lin_in + second).half().float(), wh, bias, stride=stride)
            got4 = ops.conv3d(raw_in, conv, in_affine=(a, b, False, to_act(x2), a2_, b2_))
            assert rel_err(from_act(got4), ref4) < 2e-3
    else:
        assert not (cin == 64 and k == 2)


def test_first_conv_coordconv(ops):
    for G, cout in [(16, 32), (32, 64)]:
        g = torch.Generator().manual_seed(G + cout)
        conv = torch.nn.Conv3d(4, cout, 5, 1, 2)
        occ = (torch.rand(2, 1, G, G, G, generator=g) < 0.05).float()
        occ[1] *= torch.rand(1, G, G, G, generator=g)          # non-binary values (the clip-mean input)
        ref = conv(O.add_coord_channels(occ)).detach()
        got = from_act(ops.first_conv(occ[:, 0].contiguous().cuda(), conv.cuda()))
        assert rel_err(got, ref) < 2e-3
        # GroupNorm statistics from the kernel's accumulators == statistics of the stored output
        gn = torch.nn.GroupNorm(cout // 16, cout).cuda()
        raw, a, b = ops.first_conv(occ[:, 0].contiguous().cuda(), conv, gn)
        a2, b2 = ops.gn_scale_shift(raw, gn)
        assert (a - a2).abs().max() <= 2e-3 * a2.abs().max() and (b - b2).abs().max() <= 2e-3 * (1 + b2.abs().max())


@pytest.mark.parametrize("n,cin,cout,g", [(3, 72, 48, 2), (2, 32, 64, 8), (5, 32, 32, 8), (1, 32, 64, 16)])
def test_conv_transpose(ops, n, cin, cout, g):
    gen = torch.Generator().manual_seed(3 + cin + g)
    conv = torch.nn.ConvTranspose3d(cin, cout, 2, 2)
    x = torch.randn(n, cin, g, g, g, generator=gen)
    wh = conv.weight.detach().half().float() if cin == 32 else conv.weight.detach()   # mma path: fp16 weights
    ref = F.conv_transpose3d(x.half().float(), wh, conv.bias.detach(), stride=2)
    conv = conv.cuda()
    got = from_act(ops.conv_transpose3d(to_act(x), conv))
    assert rel_err(got, ref) < 2e-3
    gn = torch.nn.GroupNorm(cout // 16, cout).cuda()
    raw, a, b = ops.conv_transpose3d(to_act(x), conv, gn)
    a2, b2 = ops.gn_scale_shift(raw, gn)
    assert torch.equal(raw, ops.conv_transpose3d(to_act(x), conv))
    assert (a - a2).abs().max() <= 2e-3 * a2.abs().max() and (b - b2).abs().max() <= 2e-3 * (1 + b2.abs().max())


# ------------------------------------------------------------------------------------------------ pointwise
@pytest.mark.parametrize("C,grid", [(32, 16), (48, 4), (64, 8), (72, 2), (128, 8), (256, 4)])
def test_groupnorm_affine(ops, C, grid):
    g = torch.Generator().manual_seed(C)
    gn = torch.nn.GroupNorm(C // 16, C)
    with torch.no_grad():
        gn.weight.copy_(1 + 0.3 * torch.randn(C, generator=g))
        gn.bias.copy_(0.3 * torch.randn(C, generator=g))
    x = torch.randn(3, C, grid, grid, grid, generator=g) * 2 + 0.7
    skip = torch.randn(3, C, grid, grid, grid, generator=g)
    xh = x.half().float()
    ref = F.leaky_relu(gn(xh), 0.01).detach()
    gn = gn.cuda()
    xa = to_act(x)
    a, b = ops.gn_scale_shift(xa, gn)
    got = from_act(ops.affine_act(xa, a, b, True))
    assert (got - ref).abs().max() < 4e-3
    ref2 = (gn.cpu()(xh) + skip.half().float()).detach()
    got2 = from_act(ops.affine_act(xa, a, b, False, x2=to_act(skip)))
    assert (got2 - ref2).abs().max() < 6e-3
    got3 = from_act(ops.affine_act(xa, a, b, False, x2=xa, a2=a, b2=b))
    assert (got3 - 2 * gn(xh).detach()).abs().max() < 8e-3


def test_upsample_trilinear(ops):
    g = torch.Generator().manual_seed(9)
    x = torch.randn(2, 64, 6, 6, 6, generator=g)
    ref = F.interpolate(x.half().float(), scale_factor=2.0, mode="trilinear", align_corners=False)
    got = from_act(ops.upsample2x(to_act(x)))
    assert (got - ref).abs().max() < 3e-3
    a = (torch.rand(2, 64, generator=g) + 0.5).cuda()
    b = torch.randn(2, 64, generator=g).cuda()
    pre = F.leaky_relu(x.half().float() * a.cpu()[:, :, None, None, None] + b.cpu()[:, :, None, None, None], 0.01)
    ref = F.interpolate(pre, scale_factor=2.0, mode="trilinear", align_corners=False)
    got = from_act(ops.upsample2x(to_act(x), a, b, act=True))
    assert (got - ref).abs().max() < 6e-3


def test_layout_roundtrip_and_mean(ops):
    g = torch.Generator().manual_seed(1)
    x = torch.randn(3, 128, 4, 4, 4, generator=g)
    assert torch.equal(ops.act_to_ncdhw(ops.ncdhw_to_act(x.cuda())).cpu(), x.half().float())
    seq = torch.rand(2, 5, 1, 8, 8, 8, generator=g)
    got = ops.mean_over_frames(seq.cuda()).cpu()
    assert (got - seq.mean(dim=1)[:, 0]).abs().max() < 1e-6


# ------------------------------------------------------------------------------------------------ heads
@pytest.mark.parametrize("g", [8, 16])
def test_heatmap_head_softargmax_render(ops, g):
    gen = torch.Generator().manual_seed(g)
    K, C, B, T = 24, 128, 2, 3
    conv1 = torch.nn.Conv3d(C, K, 1)
    prop = torch.nn.Conv3d(2, 1, 1)
    with torch.no_grad():
        conv1.weight.mul_(6.0)
        prop.weight.copy_(torch.tensor([1.5, 0.75]).view(1, 2, 1, 1, 1))
        prop.bias.fill_(-1.0)
    feat = torch.randn(B * T, C, g, g, g, generator=gen)
    prev = torch.randn(B, K, g, g, g, generator=gen)
    fh = feat.half().float()
    hm = F.leaky_relu(conv1(fh), 0.01).reshape(B * T * K, 1, g, g, g)
    pv = prev[:, None].expand(B, T, K, g, g, g).reshape(B * T * K, 1, g, g, g)
    hm = F.softplus(prop(torch.cat([hm, pv], 1))).view(B * T, K, g, g, g).detach()
    kp = O.keypoints_from_heatmap(hm)
    gs = O.render_gaussians(kp, 1.5, g)
    heat, kps, gss, hmean = ops.heatmap_head(to_act(feat), conv1.cuda(), K, 1, prev=prev.cuda(), frames_per_clip=T,
                                             prop=prop.cuda(), sigma=1.5)
    assert rel_err(heat.cpu(), hm) < 1e-4
    assert (kps.cpu() - kp).abs().max() < 2e-5
    assert (gss.cpu() - gs).abs().max() < 2e-4
    assert (hmean.cpu() - hm.mean(dim=(2, 3, 4))).abs().max() < 1e-4 * float(hm.max())
    # ST head (mode 0, C = 256)
    conv2 = torch.nn.Conv3d(256, K, 1)
    f2 = torch.randn(2, 256, g, g, g, generator=gen)
    ref = F.leaky_relu(conv2(f2.half().float()), 0.01).detach()
    got = ops.heatmap_head(to_act(f2), conv2.cuda(), K, 0)
    assert rel_err(got.cpu(), ref) < 1e-4
    # standalone render
    assert (ops.gaussian_render(kp.cuda(), 1.5, g).cpu() - gs).abs().max() < 2e-4


def test_decoder_adjust(ops):
    gen = torch.Generator().manual_seed(4)
    B, T, K, g = 2, 3, 24, 8
    conv = torch.nn.Conv3d(128 + 2 * K + 3, 128, 1)
    ff = torch.randn(B, 128, g, g, g, generator=gen)
    kp = torch.cat([torch.rand(B, T, K, 3, generator=gen) - 0.5, torch.rand(B, T, K, 1, generator=gen)], -1)
    gs = torch.stack([O.render_gaussians(kp[:, t], 1.5, g) for t in range(T)], 1)
    ffh = ff.half().float()
    ref = torch.stack([F.leaky_relu(conv(O.add_coord_channels(torch.cat([gs[:, t], ffh, gs[:, 0]], 1))), 0.01)
                       for t in range(T)], 1).detach().reshape(B * T, 128, g, g, g)
    conv = conv.cuda()
    got = from_act(ops.decoder_adjust(to_act(ff), conv, T, g, K, 1.5, keypoints=kp.reshape(B * T, K, 4).cuda()))
    assert rel_err(got, ref) < 2e-3
    got = from_act(ops.decoder_adjust(to_act(ff), conv, T, g, K, 1.5,
                                      gaussians=gs.reshape(B * T, K, g, g, g).contiguous().cuda()))
    assert rel_err(got, ref) < 2e-3


def test_final_recon_and_bce(ops):
    gen = torch.Generator().manual_seed(6)
    B, T, G, C = 2, 2, 16, 32
    gn = torch.nn.GroupNorm(2, C)
    conv = torch.nn.Conv3d(C, 1, 1)
    with torch.no_grad():
        conv.weight.mul_(4.0)
    x = torch.randn(B * T, C, G, G, G, generator=gen)
    first = (torch.rand(B, 1, G, G, G, generator=gen) < 0.1).float()
    target = (torch.rand(B * T, 1, G, G, G, generator=gen) < 0.1).float()
    xh = x.half().float()
    pre = conv(F.leaky_relu(gn(xh), 0.01))
    ff = first[:, None].expand(B, T, 1, G, G, G).reshape(B * T, 1, G, G, G)
    ref = torch.sigmoid(10.0 * (torch.tanh(pre) + ff - 0.5)).detach()
    ref_bce = F.binary_cross_entropy(ref, target, reduction="none").mean(dim=(1, 2, 3, 4))
    gn, conv = gn.cuda(), conv.cuda()
    xa = to_act(x)
    a, b = ops.gn_scale_shift(xa, gn)
    recon, bce = ops.final_recon(xa, a, b, conv, first[:, 0].contiguous().cuda(), T, 10.0, 0.5,
                                 target=target[:, 0].contiguous().cuda())
    assert (recon.cpu() - ref[:, 0]).abs().max() < 2e-2      # sigmoid slope 2.5 x fp16-rounded pre-activation
    assert (recon.cpu() - ref[:, 0]).abs().mean() < 1e-3
    assert (bce.cpu() - ref_bce).abs().max() < 2e-3 * float(ref_bce.max())


def test_scalar_parameters_by_value_and_by_device_pointer_agree(ops):
    """`bias` / (`pw0`, `pw1`, `pb`) can be passed by value or read from device memory (`bias_dev` / `prop_dev`, what the
    host wrappers use so that a training loop never synchronises on a parameter): the two routes are bit-identical."""
    from neural_marionette_b200 import _lib as L
    gen = torch.Generator().manual_seed(16)
    n, T, G, C, K, g = 4, 2, 16, 32, 24, 8
    x = to_act(torch.randn(n, C, G, G, G, generator=gen))
    a = (0.5 + torch.rand(n, C, generator=gen)).cuda()
    b = torch.randn(n, C, generator=gen).cuda()
    w = torch.randn(C, generator=gen).cuda()
    bias = torch.tensor([0.37], device="cuda")
    first = (torch.rand(n // T, G, G, G, generator=gen) < 0.1).float().cuda()
    outs = []
    for by_pointer in (False, True):
        recon = torch.empty(n, G, G, G, device="cuda")
        L.call("nm_final_recon", L.ptr(x), L.ptr(a), L.ptr(b), L.ptr(w), 0.0 if by_pointer else float(bias.item()),
               L.ptr(bias) if by_pointer else None, L.ptr(first), T, 10.0, 0.5, L.ptr(recon), None, None, None, n, G ** 3, C,
               L.stream())
        outs.append(recon)
    assert torch.equal(outs[0], outs[1])
    feat = to_act(torch.randn(n, 128, g, g, g, generator=gen))
    w1 = (torch.randn(K, 128, generator=gen) * 0.1).cuda()
    b1 = torch.randn(K, generator=gen).cuda()
    prev = torch.rand(n // T, K, g, g, g, generator=gen).cuda()
    prop = torch.tensor([0.8, 0.3, -0.1], device="cuda")
    lin = ops.linspace(g, feat.device)
    outs = []
    for by_pointer in (False, True):
        heat = torch.empty(n, K, g, g, g, device="cuda")
        kp = torch.empty(n, K, 4, device="cuda")
        pw = (0.0, 0.0, 0.0) if by_pointer else tuple(float(v) for v in prop.tolist())
        L.call("nm_heatmap_head", L.ptr(feat), L.ptr(w1), L.ptr(b1), n, g, 128, K, 1, L.ptr(prev), T, pw[0], pw[1], pw[2],
               L.ptr(prop) if by_pointer else None, L.ptr(lin), ops.gauss_width(1.5, g), L.ptr(heat), L.ptr(kp), None, None,
               L.stream())
        outs.append((heat, kp))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])


def test_chamfer(ops):
    gen = torch.Generator().manual_seed(8)
    seq = (torch.rand(2, 3, 1, 16, 16, 16, generator=gen) < 0.05).float()
    kp = torch.cat([torch.rand(2, 3, 24, 3, generator=gen) * 2 - 1, torch.rand(2, 3, 24, 1, generator=gen)], -1)
    ref = O.chamfer_vol_fit(seq, kp)
    got = ops.chamfer_vol_fit(seq.reshape(6, 16, 16, 16).cuda(), kp.reshape(6, 24, 4).cuda()).view(2, 3).cpu()
    assert (got - ref).abs().max() < 1e-5


# ------------------------------------------------------------------------------------------------ dynamics
def _dyna_setup(seed):
    import neural_marionette_b200 as nm
    hp = O.default_hparams()
    sd = O.synthetic_state_dict(hp, seed=seed)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().eval()
    net.anneal(1)
    return net, sd, hp


def test_dynamics_golden(golden_dir):
    z = np.load(os.path.join(golden_dir, "dynamics.npz"))
    net, sd, hp = _dyna_setup(int(z["seed"]))
    dm = net.dyna_module
    kp = torch.from_numpy(z["kp"]).cuda()
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        enc = dm.encode(kp, aff, eps=torch.from_numpy(np.zeros((kp.shape[1], 10, kp.shape[0], 128), np.float32)).cuda())
        assert dm.parents.cpu().tolist() == z["parents"].tolist()
        assert dm.priority.indices.cpu().tolist() == z["order"].tolist()
        assert enc["h_kypts"].shape == (3, 7, 512)
        out = dm.generate(kp[:, :3], aff, Ttot=9, Tcond=3, eps_cond=torch.from_numpy(z["eps_cond"]).cuda(),
                          eps_gen=torch.from_numpy(z["eps_gen"]).cuda())
        assert (out["keypoints_cond"].cpu() - torch.from_numpy(z["keypoints_cond"])).abs().max() < 2e-4
        assert (out["keypoints_gen"].cpu() - torch.from_numpy(z["keypoints_gen"])).abs().max() < 5e-4
        off = dm.get_offset(kp)
        assert off.shape == (3, 24, 3, 1)
        assert (off.cpu() - torch.from_numpy(z["offset"])).abs().max() < 1e-6
        flat, R = dm.extract_kypt_from_latent_and_state(torch.from_numpy(z["dec_in"]).cuda(), off)
        assert (flat.cpu() - torch.from_numpy(z["dec_flat"])).abs().max() < 2e-5
        assert (R.cpu() - torch.from_numpy(z["dec_R"])).abs().max() < 2e-5


def test_dynamics_encode_vs_oracle():
    net, sd, hp = _dyna_setup(33)
    gen = torch.Generator().manual_seed(5)
    B, T, K, Z = 5, 7, 24, 128
    kp = torch.cat([torch.rand(B, T, K, 3, generator=gen) * 1.2 - 0.6, torch.rand(B, T, K, 1, generator=gen)], -1)
    eps = torch.randn(T, 10, B, Z, generator=gen)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        got = net.dyna_module.encode(kp.cuda(), aff, eps=eps.cuda())
        ref = O.dyna_encode(kp, O.skeleton_from_affinity(aff.cpu()), sd, hp, eps=eps)
    for k in ["kypt_recon", "R", "z_kypts", "h_kypts"]:
        assert (got[k].cpu() - ref[k]).abs().max() < 5e-4, k
    assert abs(float(got["kl_kypt"]) - float(ref["kl_kypt"])) < 1e-3 * abs(float(ref["kl_kypt"]))
    assert abs(float(got["kypt_recon_loss"]) - float(ref["kypt_recon_loss"])) < 1e-3 * float(ref["kypt_recon_loss"])


def test_dynamics_large_batch_matches_small():
    """The three step kernels - a cluster of 8 CTAs per element (B <= 96), one CTA per element, one CTA per 4 elements
    (B >= 4 x #SMs) - must agree on the same elements (fp32 throughout; only the summation order differs)."""
    net, sd, hp = _dyna_setup(34)
    gen = torch.Generator().manual_seed(6)
    B, K, Z = 640, 24, 128
    kp = torch.cat([torch.rand(B, 2, K, 3, generator=gen) - 0.5, torch.rand(B, 2, K, 1, generator=gen)], -1).cuda()
    ec = torch.randn(2, 10, B, Z, generator=gen).cuda()
    eg = torch.randn(2, B, Z, generator=gen).cuda()
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        net.dyna_module.encode(kp[:2], aff)
        big = net.dyna_module.generate(kp, aff, Ttot=4, Tcond=2, eps_cond=ec, eps_gen=eg)
        mid = net.dyna_module.generate(kp[:200], aff, Ttot=4, Tcond=2, eps_cond=ec[:, :, :200].contiguous(),
                                       eps_gen=eg[:, :200].contiguous())
        small = net.dyna_module.generate(kp[:40], aff, Ttot=4, Tcond=2, eps_cond=ec[:, :, :40].contiguous(),
                                         eps_gen=eg[:, :40].contiguous())
    assert (big["keypoints_gen"][:200] - mid["keypoints_gen"]).abs().max() < 1e-5
    assert (big["keypoints_gen"][:40] - small["keypoints_gen"]).abs().max() < 1e-4
    assert (big["keypoints_cond"][:40] - small["keypoints_cond"]).abs().max() < 1e-4


def test_dynamics_interpolation_golden(golden_dir):
    """Key-frame interpolation (vis_interpolation.py:86-136) against the reference's own loop (tests/golden/interpolation.npz)."""
    z = np.load(os.path.join(golden_dir, "interpolation.npz"))
    net, sd, hp = _dyna_setup(int(z["seed"]))
    kp = torch.from_numpy(z["kp"]).cuda()
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        out = net.dyna_module.interpolate(kp, aff, sample_num=int(z["sample_num"]), sample_rate=int(z["sample_rate"]),
                                          eps=torch.from_numpy(z["eps"]).cuda())
    assert out["picks"].cpu().tolist() == z["picks"].tolist()
    assert out["keypoints"].shape == z["selected"].shape
    assert (out["keypoints"].cpu() - torch.from_numpy(z["selected"])).abs().max() < 5e-4
    # key frames return the detected keypoints themselves (with frame 0's intensities)
    assert torch.equal(out["keypoints"][0, 0, :, :3], kp[0, 0, :, :3])
    with pytest.raises(ValueError):
        net.dyna_module.interpolate(kp.repeat(2, 1, 1, 1), aff)


@pytest.mark.parametrize("n,grid,cin,cout,k", [(1, 32, 64, 32, 3), (2, 16, 32, 32, 3), (1, 16, 128, 64, 3),
                                              (2, 16, 64, 64, 3), (1, 16, 32, 64, 1)])
def test_conv3d_input_grad(ops, n, grid, cin, cout, k):
    """dL/dx of the decoder / encoder conv shapes on the forward tensor-core kernels (flipped, transposed weights)
    against torch.nn.grad.conv3d_input on the CPU (fp16-rounded operands, fp32 accumulation)."""
    g = torch.Generator().manual_seed(grid + cin + 7 * cout + k)
    conv = torch.nn.Conv3d(cin, cout, k, 1, (k - 1) // 2)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cout * k ** 3) ** 0.5)
    gy = torch.randn(n, cout, grid, grid, grid, generator=g)
    ref = torch.nn.grad.conv3d_input((n, cin, grid, grid, grid), conv.weight.detach().half().float(), gy.half().float(),
                                     padding=(k - 1) // 2)
    conv = conv.cuda()
    got = from_act(ops.conv3d_input_grad(to_act(gy), conv))
    assert got.shape == ref.shape
    assert rel_err(got, ref) < 2e-3
    # the mirrored weights follow an in-place update of the parameter (optimizer step)
    with torch.no_grad():
        conv.weight.mul_(2.0)
    assert rel_err(from_act(ops.conv3d_input_grad(to_act(gy), conv)), 2 * ref) < 2e-3


@pytest.mark.parametrize("n,grid,cin,cout", [(1, 32, 64, 32), (2, 16, 32, 32), (1, 16, 128, 64), (3, 16, 64, 64),
                                            (1, 64, 32, 32)])
def test_conv3d_weight_grad(ops, n, grid, cin, cout):
    """dL/dW of the stride-1 k3 convs against torch.nn.grad.conv3d_weight on the CPU (fp16-rounded operands, fp32
    accumulation: K = n * grid^3 products per weight -> tolerance relative to the largest gradient entry)."""
    g = torch.Generator().manual_seed(3 * grid + cin + 11 * cout)
    x = torch.randn(n, cin, grid, grid, grid, generator=g)
    gy = torch.randn(n, cout, grid, grid, grid, generator=g) / grid ** 1.5
    ref = torch.nn.grad.conv3d_weight(x.half().float(), (cout, cin, 3, 3, 3), gy.half().float(), padding=1)
    got = ops.conv3d_weight_grad(to_act(x), to_act(gy)).cpu()
    assert got.shape == ref.shape
    assert rel_err(got, ref) < 1e-3
    assert torch.equal(got, ops.conv3d_weight_grad(to_act(x), to_act(gy)).cpu())      # fixed-order split-K
    # the gather kernel computes the same tensor (any channel count that is a multiple of 8)
    alt = ops.conv3d_weight_grad(to_act(x), to_act(gy), force_gather=True).cpu()
    assert rel_err(alt, ref) < 1e-3
    got24 = ops.conv3d_weight_grad(to_act(x[:, :24]), to_act(gy)).cpu()                # Cin = 24 -> gather kernel
    assert rel_err(got24, ref[:, :24]) < 1e-3


_GNB_CASES = [(2, 16, 32, 2, True), (3, 8, 64, 4, True), (1, 32, 32, 2, False), (2, 8, 128, 8, True), (3, 4, 48, 3, True),
              (2, 2, 72, 4, False), (2, 4, 48, 3, False), (5, 2, 72, 4, True)]


@pytest.mark.parametrize("n,grid,C,groups,leaky,stats",
                         [pytest.param(*c, False, id="-".join(map(str, c))) for c in _GNB_CASES] +
                         [pytest.param(*c, True, id="-".join(map(str, c)) + "-fwdstats") for c in _GNB_CASES])
def test_groupnorm_backward(ops, n, grid, C, groups, leaky, stats):
    """dL/dx, dL/dgamma, dL/dbeta of LeakyReLU(GroupNorm(x)) against torch.autograd on the CPU (fp32 on the fp16-rounded
    tensors).  An element whose pre-activation sits within rounding of 0 may take the other LeakyReLU branch: the check
    allows 1e-5 of the elements to differ and bounds the mean error.  `stats`: x is the output of a conv3d forward and
    the backward takes the statistics that forward kept (`capture_gn_stats`), as the training step does."""
    g = torch.Generator().manual_seed(grid + C + groups)
    gn = torch.nn.GroupNorm(groups, C)
    with torch.no_grad():
        gn.weight.copy_(1 + 0.3 * torch.randn(C, generator=g))
        gn.bias.copy_(0.3 * torch.randn(C, generator=g))
    x = (torch.randn(n, C, grid, grid, grid, generator=g) * 1.5 + 0.3).half().float().requires_grad_(True)
    dz = torch.randn(n, C, grid, grid, grid, generator=g).half().float()
    gn_cuda = torch.nn.GroupNorm(groups, C).cuda()
    gn_cuda.load_state_dict(gn.state_dict())
    st = None
    if stats:
        conv = torch.nn.Conv3d(C, C, 1)
        with torch.no_grad():
            conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) * 1.5 / C ** 0.5)
            conv.bias.fill_(0.3)
        with ops.capture_gn_stats() as sink:
            raw, _, _ = ops.conv3d(to_act(x.detach()), conv.cuda(), gn_cuda)
        assert len(sink) == 1
        st = tuple(sink[0])
        x = from_act(raw).requires_grad_(True)
    y = gn(x)
    z = F.leaky_relu(y, 0.01) if leaky else y
    (z * dz).sum().backward()
    dx, dg, db, dxs = ops.groupnorm_backward(to_act(x.detach()), to_act(dz), gn_cuda, leaky=leaky, stats=st)
    dx = from_act(dx)
    # dxsum = gradient of a bias added to x (the producing conv's bias): per-channel sum of dL/dx
    ref_bias = x.grad.sum(dim=(0, 2, 3, 4))
    assert float((dxs.cpu() - ref_bias).abs().max()) <= 1e-3 * float(x.grad.abs().sum(dim=(0, 2, 3, 4)).max())
    scale = float(x.grad.abs().max())
    diff = (dx - x.grad).abs()
    assert float((diff > 3e-3 * scale).float().mean()) <= 1e-5
    assert float(diff.mean()) <= 3e-4 * scale
    assert float((dg.cpu() - gn.weight.grad).abs().max()) <= 2e-3 * float(gn.weight.grad.abs().max())
    assert float((db.cpu() - gn.bias.grad).abs().max()) <= 2e-3 * float(gn.bias.grad.abs().max())
    dx2, dg2, db2, dxs2 = ops.groupnorm_backward(to_act(x.detach()), to_act(dz), gn_cuda, leaky=leaky, stats=st)
    assert torch.equal(from_act(dx2), dx) and torch.equal(dg2, dg) and torch.equal(db2, db) and torch.equal(dxs2, dxs)
    # out_scale multiplies the fp32 outputs only
    _, dg3, db3, dxs3 = ops.groupnorm_backward(to_act(x.detach()), to_act(dz), gn_cuda, leaky=leaky, out_scale=0.25,
                                                stats=st)
    assert torch.allclose(dg3, dg * 0.25, rtol=1e-6, atol=0) and torch.allclose(db3, db * 0.25, rtol=1e-6, atol=0)
