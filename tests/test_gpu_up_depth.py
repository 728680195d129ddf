"""conv3d_k3(upsample2x(x)) with the depth half of the up-sampling applied to the accumulators (nm_conv3d_tc_up2x):
the MMAs run over the low-resolution depth and the epilogue blends the TMEM groups of neighbouring slices.  Checked
against torch (F.interpolate trilinear + F.conv3d on fp16-rounded weights), for the GroupNorm statistics of the
epilogue and for run-to-run bit identity.  Shapes are the decoder's dec.8 (64 -> 32) and dec.1 (128 -> 64, split-K) channel counts, plus depths where every slice is a border
slice (low-resolution depth 1 and 2)."""
import pytest
import torch
import torch.nn.functional as F

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


# (n, low-res D, H, W, Cin, Cout, fused GroupNorm + LeakyReLU prologue)
CASES = [
    (2, 16, 8, 8, 64, 32, True),      # dec.8 channels
    (1, 8, 16, 16, 64, 32, False),
    (3, 2, 8, 4, 64, 32, True),       # low-res depth 2: first and last slice only
    (2, 1, 8, 8, 64, 32, True),       # low-res depth 1: the first slice is the last
    (1, 4, 8, 8, 64, 64, True),       # two 32-channel parts
    (2, 8, 8, 8, 128, 64, False),     # dec.1 channels: split-K pair
    (2, 2, 16, 8, 128, 64, False),
    (3, 1, 8, 4, 128, 64, False),
]


def _setup(n, dl, hl, wl, cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    conv = torch.nn.Conv3d(cin, cout, 3, 1, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=g) / (cin * 27) ** 0.5)
        conv.bias.copy_(torch.randn(cout, generator=g))
    gn_out = torch.nn.GroupNorm(cout // 16, cout).cuda()
    raw = to_act(torch.randn(n, cin, dl, hl, wl, generator=g) * 1.5 + 0.3)
    a = (0.5 + torch.rand(n, cin, generator=g)).cuda()
    b = torch.randn(n, cin, generator=g).cuda()
    return conv.cuda(), gn_out, raw, a, b


@pytest.mark.parametrize("n,dl,hl,wl,cin,cout,fused", CASES)
def test_up2x_depth_epilogue(ops, n, dl, hl, wl, cin, cout, fused):
    conv, gn_out, raw, a, b = _setup(n, dl, hl, wl, cin, cout, seed=dl * 7 + hl + cin + cout)
    assert ops.can_conv_up2x(raw, conv)
    ia = (a, b, True) if fused else None
    act = ops.affine_act(raw, a, b, True) if fused else raw

    def run():
        out, ga, gb = ops.conv3d_up2x(raw, conv, gn_out, in_affine=ia)
        torch.cuda.synchronize()
        return out.clone(), ga.clone(), gb.clone()

    got, ga, gb = run()
    again, ga2, gb2 = run()

    ref = F.conv3d(F.interpolate(from_act(act), scale_factor=2.0, mode="trilinear", align_corners=False),
                   conv.weight.detach().cpu().half().float(), conv.bias.detach().cpu(), padding=1)
    assert rel_err(from_act(got), ref) < 3e-3
    # the epilogue's GroupNorm statistics describe the tensor it wrote
    ta, tb = ops.gn_scale_shift(got, gn_out)
    assert (ga - ta).abs().max() <= 3e-3 * ta.abs().max() and (gb - tb).abs().max() <= 3e-3 * (1 + tb.abs().max())
    # fixed reduction order: bit-identical run to run
    assert torch.equal(got, again) and torch.equal(ga, ga2) and torch.equal(gb, gb2)


def test_up2x_profile_counts_halved_flops(ops):
    """The profiling record carries the FLOPs the tensor cores execute (half of the up-sampled conv's count with the
    depth epilogue), so a layer's rate stays a hardware rate."""
    conv, _, raw, _, _ = _setup(1, 4, 8, 8, 64, 32, seed=3)
    full = 2.0 * 8 * 4 * 8 * 8 * 32 * 64 * 27
    prev = ops.PROFILE
    try:
        ops.PROFILE = {}
        ops.conv3d_up2x(raw, conv)
        torch.cuda.synchronize()
        assert [k[-1] for k in ops.PROFILE] == [full / 2]
    finally:
        ops.PROFILE = prev
