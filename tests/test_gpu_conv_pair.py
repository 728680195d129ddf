"""k3 slab convolutions on CTA pairs (W % 16 == 0) and on single CTAs (W % 16 == 8), at the detector's shapes for
G = 64 / 32 and at the edges of the pair tiling: W = 16 (one pair per row), odd batch, Cout = 128 (two 64-channel
pair-parts), non-cubic extents.  Plain, fused input GroupNorm + LeakyReLU, up-sampling, split-K (Cin = 128)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from neural_marionette_b200 import ops as _ops
    return _ops


def to_act(x):
    return x.permute(0, 2, 3, 4, 1).contiguous().half().cuda()


def from_act(y):
    return y.float().cpu().permute(0, 4, 1, 2, 3).contiguous()


def rel_err(got, ref):
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-6))


def _conv(cin, cout, g):
    conv = torch.nn.Conv3d(cin, cout, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * 27) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g))
    return conv


def _gn(cout, g):
    gn = torch.nn.GroupNorm(cout // 16, cout)
    with torch.no_grad():
        gn.weight.copy_(1 + 0.3 * torch.randn(cout, generator=g))
        gn.bias.copy_(0.3 * torch.randn(cout, generator=g))
    return gn.cuda()


# (n, D, H, W, Cin, Cout): 64^3 / 32^3 / 16^3 detector layers (Cout = 64 / 128: 64-channel pair parts, N = 192), then
# the tiling edges
PLAIN = [(1, 64, 64, 64, 32, 32), (1, 32, 32, 32, 32, 64), (2, 32, 32, 32, 64, 64), (1, 32, 32, 32, 128, 64),
         (3, 16, 16, 16, 64, 64), (2, 16, 16, 16, 64, 128), (3, 16, 16, 16, 32, 32), (1, 16, 16, 16, 64, 128),
         (1, 8, 16, 48, 32, 32), (2, 8, 16, 24, 64, 64), (1, 4, 32, 40, 32, 64)]


@pytest.mark.parametrize("n,D,H,W,cin,cout", PLAIN)
def test_slab3_plain(ops, n, D, H, W, cin, cout):
    g = torch.Generator().manual_seed(n + D + 3 * W + cin + 7 * cout)
    conv = _conv(cin, cout, g)
    x = torch.randn(n, cin, D, H, W, generator=g)
    ref = F.conv3d(x.half().float(), conv.weight.detach().half().float(), conv.bias.detach(), padding=1)
    conv = conv.cuda()
    gn = _gn(cout, g)
    raw, a, b = ops.conv3d(to_act(x), conv, gn)
    a2, b2 = ops.gn_scale_shift(raw, gn)
    torch.cuda.synchronize()
    assert rel_err(from_act(raw), ref) < 2e-3
    assert torch.equal(raw, ops.conv3d(to_act(x), conv))
    assert (a - a2).abs().max() <= 2e-3 * a2.abs().max() and (b - b2).abs().max() <= 2e-3 * (1 + b2.abs().max())


FUSED = [(1, 64, 64, 64, 32, 32), (2, 32, 32, 32, 64, 64), (3, 16, 16, 16, 64, 64), (1, 16, 16, 16, 32, 32),
         (2, 8, 16, 24, 64, 64)]


@pytest.mark.parametrize("n,D,H,W,cin,cout", FUSED)
def test_slab3_fused_input(ops, n, D, H, W, cin, cout):
    g = torch.Generator().manual_seed(11 * n + D + W + cin + cout)
    conv = _conv(cin, cout, g).cuda()
    gn = _gn(cout, g)
    raw_in = to_act(torch.randn(n, cin, D, H, W, generator=g) * 1.5 + 0.3)
    assert ops.can_fuse_input(raw_in, conv)
    a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
    b = torch.randn(n, cin, generator=g).cuda()
    act = ops.affine_act(raw_in, a, b, True)                     # separate pass (rounds to fp16)
    ref, ra, rb = ops.conv3d(act, conv, gn)
    got, ga, gb = ops.conv3d(raw_in, conv, gn, in_affine=(a, b, True))
    cpu = F.conv3d(from_act(act), conv.weight.detach().cpu().half().float(), conv.bias.detach().cpu(), padding=1)
    torch.cuda.synchronize()
    assert rel_err(from_act(got), cpu) < 2e-3
    assert rel_err(got.float().cpu(), ref.float().cpu()) < 2e-3
    assert (ga - ra).abs().max() <= 2e-3 * ra.abs().max() and (gb - rb).abs().max() <= 2e-3 * (1 + rb.abs().max())


# (n, output grid, Cin, Cout, fused): dec.8 at G = 64 / 32, dec.1 (split-K over two launches) at G = 64 / 32
UP = [(1, 64, 64, 32, True), (3, 32, 64, 32, True), (1, 32, 128, 64, False), (3, 16, 128, 64, False),
      (1, 16, 64, 64, True)]


@pytest.mark.parametrize("n,grid,cin,cout,fused", UP)
def test_slab3_upsample(ops, n, grid, cin, cout, fused):
    g = torch.Generator().manual_seed(5 * n + grid + cin + cout)
    conv = _conv(cin, cout, g).cuda()
    gn = _gn(cout, g)
    lo = grid // 2
    raw = to_act(torch.randn(n, cin, lo, lo, lo, generator=g) * 1.5 + 0.3)
    assert ops.can_conv_up2x(raw, conv)
    if fused:
        a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
        b = torch.randn(n, cin, generator=g).cuda()
        act = ops.affine_act(raw, a, b, True)
        got, ga, gb = ops.conv3d_up2x(raw, conv, gn, in_affine=(a, b, True))
    else:
        act = raw
        got, ga, gb = ops.conv3d_up2x(raw, conv, gn)
    two, ta, tb = ops.conv3d(ops.upsample2x(act), conv, gn)
    cpu = F.conv3d(F.interpolate(from_act(act), scale_factor=2.0, mode="trilinear", align_corners=False),
                   conv.weight.detach().cpu().half().float(), conv.bias.detach().cpu(), padding=1)
    torch.cuda.synchronize()
    assert rel_err(from_act(got), cpu) < 3e-3
    assert rel_err(from_act(got), from_act(two)) < 3e-3
    assert (ga - ta).abs().max() <= 3e-3 * ta.abs().max() and (gb - tb).abs().max() <= 3e-3 * (1 + tb.abs().max())
