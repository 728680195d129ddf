"""Tensor-level wrappers over the C ABI: allocate outputs with torch, launch on
the current stream.  Activations ("act") are torch.float16 channels-last tensors
of shape (n, D, H, W, C).  No CPU paths: every function requires CUDA tensors."""
from __future__ import annotations

import ctypes
import math
from typing import Optional, Tuple

import torch

from . import _lib as L

ACT_DTYPE = torch.float16
_scratch = {}
# bench.py sets this to a dict to bracket every tensor-core conv / weight-gradient launch with CUDA events on the
# launching stream: {(kind, n, grid, Cin, Cout, k, stride, flops): [(start, end), ...]}, kind = "conv" | "wgrad"
PROFILE = None


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise L.NmError("nm_b200 kernels need CUDA tensors (there is no CPU fallback)")


def workspace(nbytes: int, device, slot: str = "default") -> torch.Tensor:
    """Grow-only byte scratch per (device, slot, stream).  Kernels on one stream run in order, so a
    scratch buffer may be reused by the next launch; each stream has its own buffers."""
    key = (str(device), slot, torch.cuda.current_stream(device).cuda_stream)
    buf = _scratch.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 16), dtype=torch.uint8, device=device)
        _scratch[key] = buf
    return buf


_linspace = {}
_side_streams = {}


def side_stream(device) -> "torch.cuda.Stream":
    """One auxiliary stream per device (used to overlap the once-per-clip branch with the per-frame encoder)."""
    key = str(device)
    if key not in _side_streams:
        _side_streams[key] = torch.cuda.Stream(device=device)
    return _side_streams[key]


def linspace(n: int, device) -> torch.Tensor:
    """torch.linspace(-1, 1, n) exactly as the reference builds it (kypt_detector_utils.py:21,37,73)."""
    key = (n, str(device))
    if key not in _linspace:
        _linspace[key] = torch.linspace(-1.0, 1.0, n, device=device)
        torch.cuda.current_stream(device).synchronize()      # built once; readable from any stream afterwards
    return _linspace[key]


def gauss_width(sigma: float, g: int) -> float:
    return 2.0 * (sigma / g) ** 2.0


# ------------------------------------------------------------------ weight caches
# derived weights live OUTSIDE the modules (weak keys): `copy.deepcopy(model)` / `torch.save(model)` never see the packed
# tensors or the ctypes structs, and a collected module drops its entries
_CACHES = __import__("weakref").WeakKeyDictionary()


def _cached(module, tag: str, params, build):
    """Cache derived (packed) weights per module; rebuilt when a source parameter changes in place (load_state_dict /
    optimizer step bump ``_version``) or moves (``.cuda()``).  Edits through ``p.data`` or raw pointers do not bump
    ``_version``: call `invalidate_caches(model)` after those."""
    key = tuple((p._version, p.data_ptr(), str(p.device)) for p in params)
    slot = _CACHES.get(module)
    if slot is None:
        slot = _CACHES[module] = {}
    hit = slot.get(tag)
    if hit is None or hit[0] != key:
        with torch.no_grad():
            slot[tag] = (key, build())
    return slot[tag][1]


def packed_conv_weight(conv: torch.nn.Conv3d) -> torch.Tensor:
    def build():
        w = conv.weight.detach().float().contiguous()
        co, ci, k = w.shape[0], w.shape[1], w.shape[2]
        out = torch.empty(k ** 3, co, ci, dtype=ACT_DTYPE, device=w.device)
        L.call("nm_pack_conv_weights", L.ptr(w), L.ptr(out), co, ci, k, L.stream())
        return out
    return _cached(conv, "packed", [conv.weight], build)


def packed_pw_weight(conv: torch.nn.Conv3d) -> torch.Tensor:
    def build():
        w = conv.weight.detach().float().contiguous()
        co, ci, k = w.shape[0], w.shape[1], w.shape[2]
        out = torch.empty(L.query("nm_conv3d_pw_packed_bytes", ci, co, k), dtype=torch.uint8, device=w.device)
        L.call("nm_pack_conv_pw_weights", L.ptr(w), ci, co, k, L.ptr(out), L.stream())
        return out
    return _cached(conv, "packed_pw", [conv.weight], build)


def f32(module, name: str) -> torch.Tensor:
    p = getattr(module, name)
    return _cached(module, "f32_" + name, [p], lambda: p.detach().float().contiguous())


# ------------------------------------------------------------------ voxelize
def voxelize_points(points: torch.Tensor, grid_size: int, check: bool = True) -> torch.Tensor:
    """points (F, N, 3) float64/float32 CUDA -> (F, G, G, G) fp32 occupancy (dataset_utils.py:21-31)."""
    _need_cuda(points)
    assert points.dim() == 3 and points.shape[-1] == 3 and points.dtype in (torch.float64, torch.float32)
    points = points.contiguous()
    F, N = points.shape[:2]
    out = torch.empty(F, grid_size, grid_size, grid_size, dtype=torch.float32, device=points.device)
    flag = torch.zeros(1, dtype=torch.int32, device=points.device) if check else None
    L.call("nm_voxelize", L.ptr(points), int(points.dtype == torch.float64), F, N, grid_size, L.ptr(out),
           L.ptr(flag), L.stream())
    if check and int(flag.item()) != 0:
        raise ValueError("voxelize: point outside [-1, 1) (numpy would wrap or raise here)")
    return out


def normalize_voxelize(raw: torch.Tensor, grid_size: int, scale: float = 1.0, x_trans: float = 0.0,
                       z_trans: float = 0.0, check: bool = True) -> torch.Tensor:
    """raw (B, T, N, 3) fp32 CUDA -> (B, T, 1, G, G, G) fp32: episodic_normalization + voxelize fused."""
    _need_cuda(raw)
    assert raw.dim() == 4 and raw.shape[-1] == 3 and raw.dtype == torch.float32
    raw = raw.contiguous()
    B, T, N = raw.shape[:3]
    out = torch.empty(B, T, 1, grid_size, grid_size, grid_size, dtype=torch.float32, device=raw.device)
    ws = workspace(L.query("nm_normalize_voxelize_workspace_bytes", B), raw.device, "vox")
    flag = torch.zeros(1, dtype=torch.int32, device=raw.device) if check else None
    L.call("nm_normalize_voxelize", L.ptr(raw), B, T, N, grid_size, float(scale), float(x_trans), float(z_trans),
           L.ptr(out), None, L.ptr(ws), L.ptr(flag), L.stream())
    if check and int(flag.item()) != 0:
        raise ValueError("voxelize: point outside [-1, 1)")
    return out


# ------------------------------------------------------------------ convolutions
def _tc_ok(conv, Cin):
    k, s, Cout = conv.kernel_size[0], conv.stride[0], conv.out_channels
    return Cin % 8 == 0 and Cin >= 16 and Cout % 8 == 0 and Cout <= 256 and \
        ((s == 1 and k in (1, 3) and conv.padding[0] == (k - 1) // 2) or (s == 2 and k == 2 and conv.padding[0] == 0))


def can_fuse_input(x: torch.Tensor, conv: torch.nn.Conv3d) -> bool:
    """True when conv3d(x, conv, in_affine=...) can apply the producer's GroupNorm (+LeakyReLU) on the fly."""
    n, D, H, W, Cin = x.shape
    if _pw_ok(x, conv):
        return True
    return _tc_ok(conv, Cin) and bool(L.query("nm_conv3d_can_fuse_input", n, D, H, W, Cin, conv.out_channels,
                                              conv.kernel_size[0], conv.stride[0]))


def _pw_ok(x, conv) -> bool:
    """The memory-pipe-oriented mma.sync kernel covers this layer (Cin = 32 pool / 1x1 convs)."""
    n, D, H, W, Cin = x.shape
    k, s = conv.kernel_size[0], conv.stride[0]
    return conv.padding[0] == 0 and bool(L.query("nm_conv3d_pw_supported", n, D, H, W, Cin, conv.out_channels, k, s))


def can_fuse_input2(x: torch.Tensor, conv: torch.nn.Conv3d) -> bool:
    """True when conv3d(x, conv, in_affine=(a, b, act, x2, a2, b2)) can sum two normalised tensors on the fly."""
    n, D, H, W, Cin = x.shape
    return conv.padding[0] == 0 and bool(L.query("nm_conv3d_pw_dual_supported", n, D, H, W, Cin, conv.out_channels,
                                                 conv.kernel_size[0], conv.stride[0]))


def conv3d(x: torch.Tensor, conv: torch.nn.Conv3d, gn: Optional[torch.nn.GroupNorm] = None, in_affine=None):
    """act (n, D, H, W, Cin) -> raw conv output act (n, OD, OH, OW, Cout); bias included.
    `in_affine` = (scale, shift, act): x is the RAW output of the previous conv and act(x*scale+shift) is applied
    inside the kernel's operand path (only when can_fuse_input(x, conv)); (scale, shift, act, x2, scale2, shift2)
    additionally adds x2*scale2+shift2 (x2 as is when scale2 is None) - only when can_fuse_input2(x, conv).
    With `gn`: returns (raw, scale, shift) of the GroupNorm that follows; the statistics come out of the conv
    epilogue when the kernel supports it (no extra pass over the output), else from a reduction kernel."""
    _need_cuda(x)
    n, D, H, W, Cin = x.shape
    k, s, Cout = conv.kernel_size[0], conv.stride[0], conv.out_channels
    assert Cin == conv.in_channels and x.dtype == ACT_DTYPE and x.is_contiguous()
    if not _tc_ok(conv, Cin):
        assert in_affine is None
        out = conv3d_direct(x, conv)
        return (out,) + gn_scale_shift(out, gn) if gn is not None else out
    out = torch.empty(n, D // s, H // s, W // s, Cout, dtype=ACT_DTYPE, device=x.device)
    pointwise = _pw_ok(x, conv)
    pw, pb = packed_pw_weight(conv) if pointwise else packed_conv_weight(conv), f32(conv, "bias")
    chunks = 0
    if gn is not None:
        chunks = L.query("nm_conv3d_pw_stats_chunks" if pointwise else "nm_conv3d_stats_chunks", n, D, H, W, Cin, Cout, k, s)
    partial = None
    if chunks > 0:
        partial = workspace(n * chunks * Cout * 8, x.device, "gn").view(torch.float32)
    if PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    if pointwise:
        ia = tuple(in_affine) if in_affine is not None else (None, None, False)
        ia = ia + (None, None, None) if len(ia) == 3 else ia
        assert ia[3] is None or (ia[3].shape == x.shape and ia[3].is_contiguous())
        L.call("nm_conv3d_pw", L.ptr(x), L.ptr(pw), L.ptr(pb), L.ptr(out), n, D, H, W, Cin, Cout, k, s,
               L.ptr(ia[0]), L.ptr(ia[1]), int(ia[2]), L.ptr(ia[3]), L.ptr(ia[4]), L.ptr(ia[5]), L.ptr(partial),
               L.stream())
    elif in_affine is None:
        L.call("nm_conv3d_tc", L.ptr(x), L.ptr(pw), L.ptr(pb), L.ptr(out), n, D, H, W, Cin, Cout, k, s,
               L.ptr(partial), L.stream())
    else:
        L.call("nm_conv3d_tc_fused", L.ptr(x), L.ptr(pw), L.ptr(pb), L.ptr(out), n, D, H, W, Cin, Cout, k, s,
               L.ptr(in_affine[0]), L.ptr(in_affine[1]), int(in_affine[2]), L.ptr(partial), L.stream())
    if PROFILE is not None:
        e1.record()
        flops = 2.0 * n * (D // s) * (H // s) * (W // s) * Cout * Cin * k ** 3
        PROFILE.setdefault(("conv", n, D, Cin, Cout, k, s, flops), []).append((e0, e1))
    if gn is None:
        return out
    if chunks == 0:
        return (out,) + gn_scale_shift(out, gn)
    a, b = _gn_finalize(partial, n, out.numel() // (n * Cout), Cout, gn, chunks, x.device)
    return out, a, b


def can_conv_up2x(x_lo: torch.Tensor, conv: torch.nn.Conv3d) -> bool:
    n, D, H, W, Cin = x_lo.shape
    return conv.kernel_size[0] == 3 and conv.stride[0] == 1 and conv.padding[0] == 1 and \
        bool(L.query("nm_conv3d_up2x_supported", n, 2 * D, 2 * H, 2 * W, Cin, conv.out_channels))


# ------------------------------------------------------------------ backward bricks (config #4 training step)
# Activation gradients are fp16 tensors multiplied by a loss scale; every fp32 output (parameter / keypoint
# gradients) is divided by it inside the kernels.  `ConvGNFinalRecon.backward` (autograd.py) picks the scale of a
# backward pass from the incoming loss gradient; the other backward functions read it from here.
_GRAD_SCALE = [4096.0]


def grad_scale() -> float:
    return _GRAD_SCALE[0]


def set_grad_scale(value: float) -> None:
    _GRAD_SCALE[0] = float(value)


class _ConvSpec:
    """What conv3d / conv_transpose3d read of an nn.Conv3d / nn.ConvTranspose3d, for the derived (mirrored) convolutions of
    the backward: built on the device from the live weight - no host-side module construction, no host -> device copy
    (the mirrors are rebuilt after every optimizer step)."""

    def __init__(self, transposed, cin, cout, k, stride, weight):
        pad = (k - 1) // 2 if stride == 1 else 0
        self.transposed = transposed
        self.in_channels, self.out_channels = cin, cout
        self.kernel_size, self.stride, self.padding = (k, k, k), (stride, stride, stride), (pad, pad, pad)
        self.output_padding, self.groups = (0, 0, 0), 1
        self.weight = weight.detach().float().contiguous()
        self.bias = torch.zeros(cout, dtype=torch.float32, device=weight.device)


def _zero_bias_mirror(kind, cin, cout, k, stride, weight):
    return _ConvSpec(kind == "convT", cin, cout, k, stride, weight)


def conv3d_input_grad(grad_out: torch.Tensor, conv: torch.nn.Conv3d) -> torch.Tensor:
    """dL/dx of an nn.Conv3d of the detector.  Stride-1 "same" convs (k = 1 or 3): the conv of dL/dy with the
    spatially flipped taps and the in / out channels swapped, on the forward tensor-core kernels.  k2/s2 "pool" convs:
    the transposed convolution with the same weight tensor.  grad_out act (n, OD, OH, OW, Cout) -> act (n, D, H, W, Cin)."""
    k, s = conv.kernel_size[0], conv.stride[0]
    if conv.groups != 1:
        raise NotImplementedError("conv3d_input_grad: groups != 1")
    if s == 1 and k in (1, 3) and conv.padding[0] == (k - 1) // 2:
        mirror = _cached(conv, "dgrad_mirror", [conv.weight], lambda: _zero_bias_mirror(
            "conv", conv.out_channels, conv.in_channels, k, 1, conv.weight.detach().flip(2, 3, 4).transpose(0, 1)))
        return conv3d(grad_out, mirror)
    if s == 2 and k == 2 and conv.padding[0] == 0 and conv.in_channels >= 64 and conv.in_channels % 8 == 0 and \
            conv.out_channels >= 16 and conv.out_channels % 8 == 0:
        # wide layers: the transposed conv as 1x1 convs dL/dy -> (tap, ci) on the tensor cores + a depth-to-space scatter
        Co, Ci = conv.out_channels, conv.in_channels
        tp = max(1, min(8, 256 // Ci))                                     # taps per 1x1 conv (N = tp * Ci <= 256)

        def build():
            w = conv.weight.detach().reshape(Co, Ci, 8).permute(2, 1, 0)   # [tap][ci][co]
            return [_zero_bias_mirror("conv", Co, tp * Ci, 1, 1, w[t0:t0 + tp].reshape(tp * Ci, Co, 1, 1, 1))
                    for t0 in range(0, 8, tp)]
        mirrors = _cached(conv, "dgrad_mirror_1x1", [conv.weight], build)
        n, D, H, W, _ = grad_out.shape
        dx = torch.empty(n, 2 * D, 2 * H, 2 * W, Ci, dtype=ACT_DTYPE, device=grad_out.device)
        for j, m in enumerate(mirrors):
            y = conv3d(grad_out, m)
            L.call("nm_depth_to_space2", L.ptr(y), L.ptr(dx), n, D, H, W, Ci, j * tp, tp, L.stream())
        return dx
    if s == 2 and k == 2 and conv.padding[0] == 0:
        # weight (Cout, Cin, 2, 2, 2) read as the (in = Cout, out = Cin) weight of a ConvTranspose3d
        mirror = _cached(conv, "dgrad_mirror", [conv.weight], lambda: _zero_bias_mirror(
            "convT", conv.out_channels, conv.in_channels, 2, 2, conv.weight.detach()))
        return conv_transpose3d(grad_out, mirror)
    raise NotImplementedError("conv3d_input_grad: stride-1 'same' convolutions with k in (1, 3) or k2/s2 only")


def conv_transpose3d_input_grad(grad_out: torch.Tensor, conv: torch.nn.ConvTranspose3d) -> torch.Tensor:
    """dL/dx of nn.ConvTranspose3d(k2, s2): the k2/s2 convolution of dL/dy with the same weight tensor read as
    (out = Cin, in = Cout, 2, 2, 2).  grad_out act (n, 2D, 2H, 2W, Cout) -> act (n, D, H, W, Cin)."""
    mirror = _cached(conv, "dgrad_mirror", [conv.weight], lambda: _zero_bias_mirror(
        "conv", conv.out_channels, conv.in_channels, 2, 2, conv.weight.detach()))
    return conv3d(grad_out, mirror)


def _slab_wgrad_ok(x, Cout) -> bool:
    n, D, H, W, Cin = x.shape
    return Cin % 32 == 0 and Cout % 32 == 0 and Cin <= 256 and Cout <= 256 and W in (16, 32, 48, 64)


def conv3d_weight_grad(x: torch.Tensor, grad_out: torch.Tensor, k: int = 3, stride: int = 1,
                       out_scale: float = 1.0, force_gather: bool = False, impl: Optional[str] = None) -> torch.Tensor:
    """dL/dW of an nn.Conv3d ((k, stride) in {(1, 1), (3, 1), (2, 2)}): x act (n, D, H, W, Cin), grad_out act
    (n, OD, OH, OW, Cout) -> (Cout, Cin, k, k, k) fp32, multiplied by out_scale.  The k3 layers go to the tcgen05
    kernel where it covers the shape (`impl`: "tc" | "slab" | "gather" forces a kernel - tests)."""
    _need_cuda(x, grad_out)
    n, D, H, W, Cin = x.shape
    Cout = grad_out.shape[-1]
    assert x.dtype == ACT_DTYPE and grad_out.dtype == ACT_DTYPE and x.is_contiguous() and grad_out.is_contiguous()
    assert tuple(grad_out.shape[1:4]) == (D // stride, H // stride, W // stride) and grad_out.shape[0] == n
    dw = torch.empty(Cout, Cin, k, k, k, dtype=torch.float32, device=x.device)
    if force_gather:
        impl = "gather"
    tc_ok = k == 3 and stride == 1 and bool(L.query("nm_conv3d_k3_wgrad_tc_supported", n, D, H, W, Cin, Cout))
    if impl == "tc" or (impl is None and tc_ok):
        nbytes = L.query("nm_conv3d_k3_wgrad_tc_workspace_bytes", n, D, H, W, Cin, Cout)
        ws = workspace(max(nbytes, 16), x.device, "wgrad")
        if PROFILE is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        L.call("nm_conv3d_k3_wgrad_tc", L.ptr(x), L.ptr(grad_out), n, D, H, W, Cin, Cout, float(out_scale), L.ptr(dw),
               L.ptr(ws), L.stream())
        if PROFILE is not None:
            e1.record()
            PROFILE.setdefault(("wgrad", n, D, Cin, Cout, 3, 1, 2.0 * n * D * H * W * Cout * Cin * 27), []).append((e0, e1))
        return dw
    if k == 3 and stride == 1 and _slab_wgrad_ok(x, Cout) and impl != "gather":
        nbytes = L.query("nm_conv3d_k3_wgrad_workspace_bytes", n, D, H, W, Cin, Cout)
        ws = workspace(max(nbytes, 16), x.device, "wgrad")
        L.call("nm_conv3d_k3_wgrad", L.ptr(x), L.ptr(grad_out), n, D, H, W, Cin, Cout, float(out_scale), L.ptr(dw),
               L.ptr(ws), L.stream())
        return dw
    OD, OH, OW = grad_out.shape[1:4]
    nbytes = L.query("nm_conv3d_wgrad_gather_workspace_bytes", n, OD, OH, OW, Cout, Cin, k, stride)
    ws = workspace(max(nbytes, 16), x.device, "wgrad")
    L.call("nm_conv3d_wgrad_gather", L.ptr(grad_out), L.ptr(x), n, OD, OH, OW, Cout, Cin, k, stride, float(out_scale),
           L.ptr(dw), L.ptr(ws), L.stream())
    return dw


def conv_transpose3d_weight_grad(x: torch.Tensor, grad_out: torch.Tensor, out_scale: float = 1.0) -> torch.Tensor:
    """dL/dW of nn.ConvTranspose3d(k2, s2): x act (n, D, H, W, Cin), grad_out act (n, 2D, 2H, 2W, Cout) ->
    (Cin, Cout, 2, 2, 2) fp32, multiplied by out_scale."""
    _need_cuda(x, grad_out)
    n, D, H, W, Cin = x.shape
    Cout = grad_out.shape[-1]
    assert tuple(grad_out.shape[:4]) == (n, 2 * D, 2 * H, 2 * W) and x.is_contiguous() and grad_out.is_contiguous()
    dw = torch.empty(Cin, Cout, 2, 2, 2, dtype=torch.float32, device=x.device)
    nbytes = L.query("nm_conv3d_wgrad_gather_workspace_bytes", n, D, H, W, Cin, Cout, 2, 2)
    ws = workspace(max(nbytes, 16), x.device, "wgrad")
    L.call("nm_conv3d_wgrad_gather", L.ptr(x), L.ptr(grad_out), n, D, H, W, Cin, Cout, 2, 2, float(out_scale), L.ptr(dw),
           L.ptr(ws), L.stream())
    return dw


def groupnorm_backward(x: torch.Tensor, grad_out: torch.Tensor, gn: torch.nn.GroupNorm, leaky: bool = True,
                       out_scale: float = 1.0, stats=None):
    """Backward of LeakyReLU(GroupNorm(x)) (`leaky`) or GroupNorm(x): x, grad_out act (n, D, H, W, C) ->
    (grad_in act, dgamma (C), dbeta (C), dxsum (C)) - the fp32 outputs multiplied by out_scale; dxsum = sum of grad_in
    over samples and voxels = gradient of the bias of the conv that produced x.  `stats` = (mean_rstd, xsum) kept from the
    forward (`capture_gn_stats`) skips the statistics pass over x."""
    _need_cuda(x, grad_out)
    assert x.shape == grad_out.shape and x.dtype == ACT_DTYPE and grad_out.dtype == ACT_DTYPE
    assert x.is_contiguous() and grad_out.is_contiguous()
    n, C = x.shape[0], x.shape[-1]
    S = x.numel() // (n * C)
    dx = torch.empty_like(x)
    dg = torch.empty(C, dtype=torch.float32, device=x.device)
    db = torch.empty(C, dtype=torch.float32, device=x.device)
    dxs = torch.empty(C, dtype=torch.float32, device=x.device)
    ws = workspace(max(L.query("nm_groupnorm_backward_workspace_bytes", n, C, gn.num_groups), 16), x.device, "gnb")
    mr, xs = stats if stats is not None else (None, None)
    L.call("nm_groupnorm_backward", L.ptr(x), L.ptr(grad_out), L.ptr(f32(gn, "weight")), L.ptr(f32(gn, "bias")), n, S, C,
           gn.num_groups, float(gn.eps), int(leaky), float(out_scale), L.ptr(mr), L.ptr(xs), L.ptr(dx), L.ptr(dg),
           L.ptr(db), L.ptr(dxs), L.ptr(ws), L.stream())
    return dx, dg, db, dxs


def upsample2x_backward(grad_out: torch.Tensor) -> torch.Tensor:
    """Backward of upsample2x without prologue: act (n, 2D, 2H, 2W, C) -> act (n, D, H, W, C)."""
    _need_cuda(grad_out)
    n, D2, H2, W2, C = grad_out.shape
    assert grad_out.dtype == ACT_DTYPE and grad_out.is_contiguous()
    dx = torch.empty(n, D2 // 2, H2 // 2, W2 // 2, C, dtype=ACT_DTYPE, device=grad_out.device)
    ws = workspace(L.query("nm_upsample2x_backward_workspace_bytes", n, D2 // 2, H2 // 2, W2 // 2, C), grad_out.device, "up_bwd")
    L.call("nm_upsample2x_backward", L.ptr(grad_out), L.ptr(dx), n, D2 // 2, H2 // 2, W2 // 2, C, L.ptr(ws), L.stream())
    return dx


def first_conv_weight_grad(occ: torch.Tensor, grad_out: torch.Tensor, out_scale: float = 1.0) -> torch.Tensor:
    """dL/dW of the CoordConv first layer: occ (n, G, G, G) fp32, grad_out act (n, G, G, G, Cout) -> (Cout, 4, 5, 5, 5)."""
    _need_cuda(occ, grad_out)
    n, G = occ.shape[0], occ.shape[1]
    Cout = grad_out.shape[-1]
    assert occ.dtype == torch.float32 and occ.is_contiguous() and grad_out.is_contiguous()
    dw = torch.empty(Cout, 4, 5, 5, 5, dtype=torch.float32, device=occ.device)
    ws = workspace(L.query("nm_first_conv_wgrad_workspace_bytes", n, Cout), occ.device, "wgrad")
    L.call("nm_first_conv_wgrad", L.ptr(occ), L.ptr(grad_out), L.ptr(linspace(G, occ.device)), n, G, Cout,
           float(out_scale), L.ptr(dw), L.ptr(ws), L.stream())
    return dw


def final_recon_backward(raw, a, b, conv: torch.nn.Conv3d, first_frame, frames_per_clip, sharpness, translation,
                         recon, target, grad_bce, scale: float):
    """-> (grad_act act (n, D, H, W, C) times `scale`, dw (1, C, 1, 1, 1), dbias (1))."""
    n, D, H, W, C = raw.shape
    S = D * H * W
    w = f32(conv, "weight").reshape(-1)
    bias_dev = f32(conv, "bias")                       # the live parameter, read on the device (no host sync per step)
    dact = torch.empty_like(raw)
    dw = torch.empty(1, C, 1, 1, 1, dtype=torch.float32, device=raw.device)
    db = torch.empty(1, dtype=torch.float32, device=raw.device)
    ws = workspace(L.query("nm_final_recon_backward_workspace_bytes", n), raw.device, "recon_bwd")
    L.call("nm_final_recon_backward", L.ptr(raw), L.ptr(a), L.ptr(b), L.ptr(w), 0.0, L.ptr(bias_dev), L.ptr(first_frame), frames_per_clip,
           float(sharpness), float(translation), L.ptr(recon), L.ptr(target), L.ptr(grad_bce), float(scale), L.ptr(dact),
           L.ptr(dw), L.ptr(db), L.ptr(ws), n, S, C, L.stream())
    return dact, dw, db


def final_recon_backward_fused(raw, a, b, conv: torch.nn.Conv3d, gn: torch.nn.GroupNorm, stats, sharpness, recon, target,
                               grad_bce, scale: float):
    """Decoder tail backward fused with the GroupNorm + LeakyReLU in front of it: -> (grad_raw act times `scale`,
    dw14 (1, C, 1, 1, 1), db14 (1), dgamma (C), dbeta (C), dxsum (C) = bias gradient of the conv that produced `raw`)."""
    n, D, H, W, C = raw.shape
    S = D * H * W
    dev = raw.device
    w = f32(conv, "weight").reshape(-1)
    bias_dev = f32(conv, "bias")
    draw = torch.empty_like(raw)
    dw = torch.empty(1, C, 1, 1, 1, dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    dg, dbeta, dxs = (torch.empty(C, dtype=torch.float32, device=dev) for _ in range(3))
    ws = workspace(L.query("nm_final_recon_backward_fused_workspace_bytes", n, S, C, gn.num_groups), dev, "recon_bwd")
    mr, xs = stats
    L.call("nm_final_recon_backward_fused", L.ptr(raw), L.ptr(a), L.ptr(b), L.ptr(w), 0.0, L.ptr(bias_dev), float(sharpness), L.ptr(recon),
           L.ptr(target), L.ptr(grad_bce), float(scale), L.ptr(f32(gn, "weight")), L.ptr(f32(gn, "bias")), L.ptr(mr), L.ptr(xs),
           gn.num_groups, L.ptr(draw), L.ptr(dw), L.ptr(db), L.ptr(dg), L.ptr(dbeta), L.ptr(dxs), L.ptr(ws), n, S, C, L.stream())
    return draw, dw, db, dg, dbeta, dxs


def heatmap_head_backward(feature, conv1: torch.nn.Conv3d, K: int, mode: int, scale: float, prev=None,
                          frames_per_clip: int = 1, prop: Optional[torch.nn.Conv3d] = None, heat=None, keypoints=None,
                          heat_mean=None, grad_keypoints=None, grad_heat_mean=None, grad_heat=None, dq_in=None):
    """Backward of heatmap_head.  mode 1 -> (grad_feature act, dq (n, K, g, g, g), dw1, db1, dprop (3));
    mode 0 -> (grad_feature act, None, dw1, db1, None)."""
    n, g, C = feature.shape[0], feature.shape[1], feature.shape[-1]
    dev = feature.device
    w1 = f32(conv1, "weight").reshape(K, C)
    b1 = f32(conv1, "bias")
    dfeat = torch.empty_like(feature)
    dw1 = torch.empty(K, C, 1, 1, 1, dtype=torch.float32, device=dev)
    db1 = torch.empty(K, dtype=torch.float32, device=dev)
    ws = workspace(L.query("nm_heatmap_head_backward_workspace_bytes", n, C, K), dev, "head_bwd")
    prop_dev = None                                     # (pw0, pw1, pb) are read on the device
    if mode == 1:
        prop_dev = _prop_dev(prop)
        dq = torch.empty(n, K, g, g, g, dtype=torch.float32, device=dev)
        dprop = torch.empty(3, dtype=torch.float32, device=dev)
    else:
        dq, dprop = None, None
        if dq_in is not None:
            prop_dev = _prop_dev(prop)                  # mode 0 only uses pw1
    L.call("nm_heatmap_head_backward", L.ptr(feature), L.ptr(w1), L.ptr(b1), n, g, C, K, mode, L.ptr(prev),
           frames_per_clip, 0.0, 0.0, 0.0, L.ptr(prop_dev), L.ptr(linspace(g, dev)), L.ptr(heat), L.ptr(keypoints), L.ptr(heat_mean),
           L.ptr(grad_keypoints), L.ptr(grad_heat_mean), L.ptr(grad_heat), L.ptr(dq_in), float(scale), L.ptr(dfeat),
           L.ptr(dq), L.ptr(dw1), L.ptr(db1), L.ptr(dprop), L.ptr(ws), L.stream())
    return dfeat, dq, dw1, db1, dprop


def decoder_adjust_backward(grad_out, out, ff_act, keypoints, conv: torch.nn.Conv3d, frames_per_clip: int, g: int, K: int,
                            sigma: float, scale: float):
    """-> (grad_first_feature act (B, g, g, g, 128) times scale, grad_keypoints (n, K, 4), dweight, dbias)."""
    B = ff_act.shape[0]
    n = B * frames_per_clip
    dev = ff_act.device
    dff = torch.empty_like(ff_act)
    dkp = torch.empty(n, K, 4, dtype=torch.float32, device=dev)
    dw = torch.empty(conv.out_channels, conv.in_channels, 1, 1, 1, dtype=torch.float32, device=dev)
    db = torch.empty(conv.out_channels, dtype=torch.float32, device=dev)
    ws = workspace(L.query("nm_decoder_adjust_backward_workspace_bytes", B, frames_per_clip), dev, "adjust_bwd")
    w = f32(conv, "weight").reshape(conv.out_channels, -1)
    L.call("nm_decoder_adjust_backward", L.ptr(grad_out), L.ptr(out), L.ptr(ff_act), L.ptr(keypoints), L.ptr(w), B,
           frames_per_clip, g, K, L.ptr(linspace(g, dev)), gauss_width(sigma, g), float(scale), L.ptr(dff), L.ptr(dkp),
           L.ptr(dw), L.ptr(db), L.ptr(ws), L.stream())
    return dff, dkp, dw, db


def chamfer_vol_fit_backward(seq_frames: torch.Tensor, keypoints: torch.Tensor, grad_out: torch.Tensor) -> torch.Tensor:
    """-> grad_keypoints (n, K, 4) fp32."""
    n, G = seq_frames.shape[0], seq_frames.shape[-1]
    K = keypoints.shape[1]
    dkp = torch.empty(n, K, 4, dtype=torch.float32, device=seq_frames.device)
    ws = workspace(L.query("nm_chamfer_vol_fit_backward_workspace_bytes", n, K), seq_frames.device, "chamfer_bwd")
    L.call("nm_chamfer_vol_fit_backward", L.ptr(seq_frames), L.ptr(keypoints), L.ptr(linspace(G, seq_frames.device)),
           L.ptr(grad_out), n, K, G, L.ptr(dkp), L.ptr(ws), L.stream())
    return dkp


def invalidate_caches(module: torch.nn.Module) -> None:
    """Drop every derived (packed / transposed) weight cached on the sub-modules: call after editing parameters through
    `.data` or raw pointers (the fused optimizer does), which does not bump `Tensor._version`."""
    for m in module.modules():
        _CACHES.pop(m, None)


def conv3d_up2x(x_lo: torch.Tensor, conv: torch.nn.Conv3d, gn: Optional[torch.nn.GroupNorm] = None, in_affine=None):
    """conv3d_k3(upsample2x_trilinear(act(x_lo*scale+shift))) without materialising the up-sampled tensor.
    x_lo act (n, D, H, W, Cin) -> raw (n, 2D, 2H, 2W, Cout) [, GroupNorm scale, shift]."""
    _need_cuda(x_lo)
    n, D, H, W, Cin = x_lo.shape
    Cout = conv.out_channels
    assert can_conv_up2x(x_lo, conv) and x_lo.dtype == ACT_DTYPE and x_lo.is_contiguous()
    out = torch.empty(n, 2 * D, 2 * H, 2 * W, Cout, dtype=ACT_DTYPE, device=x_lo.device)
    pw, pb = packed_conv_weight(conv), f32(conv, "bias")
    chunks = L.query("nm_conv3d_stats_chunks", n, 2 * D, 2 * H, 2 * W, Cin, Cout, 3, 1) if gn is not None else 0
    partial = workspace(n * chunks * Cout * 8, x_lo.device, "gn").view(torch.float32) if chunks else None
    ia = in_affine if in_affine is not None else (None, None, False)
    if PROFILE is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    L.call("nm_conv3d_tc_up2x", L.ptr(x_lo), L.ptr(pw), L.ptr(pb), L.ptr(out), n, 2 * D, 2 * H, 2 * W, Cin, Cout,
           L.ptr(ia[0]), L.ptr(ia[1]), int(ia[2]), L.ptr(partial), L.stream())
    if PROFILE is not None:
        e1.record()
        # what the tensor cores execute: the depth half of the up-sampling is applied to the accumulators (MMAs over
        # the D low-resolution slices)
        flops = 2.0 * n * 8 * D * H * W * Cout * Cin * 27 / 2
        PROFILE.setdefault(("conv", n, 2 * D, Cin, Cout, 3, 1, flops), []).append((e0, e1))
    if gn is None:
        return out
    a, b = _gn_finalize(partial, n, 8 * D * H * W, Cout, gn, chunks, x_lo.device)
    return out, a, b


def conv3d_direct(x: torch.Tensor, conv: torch.nn.Conv3d) -> torch.Tensor:
    """CUDA-core cross-check of conv3d (tests only)."""
    n, D, H, W, Cin = x.shape
    k, s, pad, Cout = conv.kernel_size[0], conv.stride[0], conv.padding[0], conv.out_channels
    out = torch.empty(n, (D + 2 * pad - k) // s + 1, (H + 2 * pad - k) // s + 1, (W + 2 * pad - k) // s + 1, Cout,
                      dtype=ACT_DTYPE, device=x.device)
    L.call("nm_conv3d_direct", L.ptr(x), L.ptr(f32(conv, "weight")), L.ptr(f32(conv, "bias")), L.ptr(out),
           n, D, H, W, Cin, Cout, k, s, pad, L.stream())
    return out


def conv_transpose3d(x: torch.Tensor, conv: torch.nn.ConvTranspose3d, gn: Optional[torch.nn.GroupNorm] = None):
    """ConvTranspose3d(k2, s2): act (n, D, H, W, Cin) -> raw (n, 2D, 2H, 2W, Cout) [, GroupNorm scale, shift]."""
    n, D, H, W, Cin = x.shape
    Cout = conv.out_channels
    assert conv.kernel_size[0] == 2 and conv.stride[0] == 2 and tuple(conv.output_padding) == (0, 0, 0), \
        "only ConvTranspose3d(k2, s2, output_padding 0) is implemented (grid sizes divisible by 32)"
    out = torch.empty(n, 2 * D, 2 * H, 2 * W, Cout, dtype=ACT_DTYPE, device=x.device)
    if L.query("nm_conv_transpose3d_pw_supported", n, D, H, W, Cin, Cout):
        def build():
            t = torch.empty(L.query("nm_conv_transpose3d_pw_packed_bytes", Cin, Cout), dtype=torch.uint8, device=x.device)
            L.call("nm_pack_conv_transpose3d_pw_weights", L.ptr(conv.weight.detach().float().contiguous()), Cin, Cout,
                   L.ptr(t), L.stream())
            return t
        pw = _cached(conv, "packed_pwT", [conv.weight], build)
        chunks = L.query("nm_conv_transpose3d_pw_stats_chunks", n, D, H, W, Cin, Cout) if gn is not None else 0
        partial = workspace(n * chunks * Cout * 8, x.device, "gn").view(torch.float32) if chunks else None
        L.call("nm_conv_transpose3d_pw", L.ptr(x), L.ptr(pw), L.ptr(f32(conv, "bias")), L.ptr(out), n, D, H, W, Cin,
               Cout, L.ptr(partial), L.stream())
        if gn is None:
            return out
        a, b = _gn_finalize(partial, n, 8 * D * H * W, Cout, gn, chunks, x.device)
        return out, a, b
    wt = _cached(conv, "tapmajor", [conv.weight],
                 lambda: conv.weight.detach().float().permute(2, 3, 4, 0, 1).reshape(8, Cin, Cout).contiguous())
    L.call("nm_conv_transpose3d_k2s2", L.ptr(x), L.ptr(wt), L.ptr(f32(conv, "bias")), L.ptr(out),
           n, D, H, W, Cin, Cout, L.stream())
    return (out,) + gn_scale_shift(out, gn) if gn is not None else out


def first_conv(occ: torch.Tensor, conv: torch.nn.Conv3d, gn: Optional[torch.nn.GroupNorm] = None):
    """occ (n, G, G, G) fp32 -> act (n, G, G, G, Cout): CoordConv k5 layer with analytic coordinate channels.
    With `gn`: returns (raw, scale, shift) of the GroupNorm that follows, statistics from the kernel's accumulators."""
    _need_cuda(occ)
    n, G = occ.shape[0], occ.shape[1]
    Cout = conv.out_channels
    assert conv.in_channels == 4 and conv.kernel_size[0] == 5 and occ.dtype == torch.float32 and occ.is_contiguous()

    def build():
        t = torch.empty(L.query("nm_first_conv_tables_bytes", Cout), dtype=torch.uint8, device=occ.device)
        L.call("nm_first_conv_prepare", L.ptr(conv.weight.detach().float().contiguous()), Cout, L.ptr(t), L.stream())
        return t
    tables = _cached(conv, "first_tables", [conv.weight], build)
    out = torch.empty(n, G, G, G, Cout, dtype=ACT_DTYPE, device=occ.device)
    chunks = L.query("nm_first_conv_stats_chunks", G) if gn is not None else 0
    partial = workspace(n * chunks * Cout * 8, occ.device, "gn").view(torch.float32) if chunks else None
    L.call("nm_first_conv_k5", L.ptr(occ), L.ptr(tables), L.ptr(f32(conv, "bias")), L.ptr(linspace(G, occ.device)),
           n, G, Cout, L.ptr(out), L.ptr(partial), L.stream())
    if gn is None:
        return out
    a, b = _gn_finalize(partial, n, G ** 3, Cout, gn, chunks, occ.device)
    return out, a, b


# ------------------------------------------------------------------ GroupNorm / pointwise
# The training path keeps the forward's GroupNorm statistics for the backward (mean / rstd per (sample, group) and the
# per-(sample, channel) sums), so that nm_groupnorm_backward skips its statistics pass: inside `capture_gn_stats()` every
# GroupNorm finalize of this module appends (mean_rstd (n, groups, 2), xsum (n, C)) to the yielded list.
_GN_SINK = [None]


@__import__("contextlib").contextmanager
def capture_gn_stats():
    prev, sink = _GN_SINK[0], []
    _GN_SINK[0] = sink
    try:
        yield sink
    finally:
        _GN_SINK[0] = prev


def _gn_stat_outputs(n, C, groups, device):
    if _GN_SINK[0] is None:
        return None, None
    mr = torch.empty(n, groups, 2, dtype=torch.float32, device=device)
    xs = torch.empty(n, C, dtype=torch.float32, device=device)
    _GN_SINK[0].append((mr, xs))
    return mr, xs


def _gn_finalize(partial, n, S, C, gn, chunks, device):
    """scale / shift (n, C) of the GroupNorm from the partial statistics a conv epilogue produced."""
    a = torch.empty(n, C, dtype=torch.float32, device=device)
    b = torch.empty_like(a)
    mr, xs = _gn_stat_outputs(n, C, gn.num_groups, device)
    L.call("nm_groupnorm_finalize", L.ptr(partial), n, S, C, gn.num_groups, chunks, L.ptr(f32(gn, "weight")),
           L.ptr(f32(gn, "bias")), float(gn.eps), L.ptr(a), L.ptr(b), L.ptr(mr), L.ptr(xs), L.stream())
    return a, b


def gn_scale_shift(raw: torch.Tensor, gn: torch.nn.GroupNorm) -> Tuple[torch.Tensor, torch.Tensor]:
    n, C = raw.shape[0], raw.shape[-1]
    S = raw.numel() // (n * C)
    a = torch.empty(n, C, dtype=torch.float32, device=raw.device)
    b = torch.empty_like(a)
    mr, xs = _gn_stat_outputs(n, C, gn.num_groups, raw.device)
    ws = workspace(L.query("nm_gn_workspace_bytes", n, S, C), raw.device, "gn")
    L.call("nm_groupnorm_scale_shift", L.ptr(raw), n, S, C, gn.num_groups, L.ptr(f32(gn, "weight")),
           L.ptr(f32(gn, "bias")), float(gn.eps), L.ptr(a), L.ptr(b), L.ptr(ws), L.ptr(mr), L.ptr(xs), L.stream())
    return a, b


def affine_act(x1, a1, b1, act: bool, x2=None, a2=None, b2=None) -> torch.Tensor:
    n, C = x1.shape[0], x1.shape[-1]
    S = x1.numel() // (n * C)
    out = torch.empty_like(x1)
    L.call("nm_affine_act", L.ptr(x1), L.ptr(a1), L.ptr(b1), int(act), L.ptr(x2), L.ptr(a2), L.ptr(b2), L.ptr(out),
           n, S, C, L.stream())
    return out


def upsample2x(x, a=None, b=None, act: bool = False) -> torch.Tensor:
    n, D, H, W, C = x.shape
    out = torch.empty(n, 2 * D, 2 * H, 2 * W, C, dtype=ACT_DTYPE, device=x.device)
    L.call("nm_upsample2x", L.ptr(x), L.ptr(a), L.ptr(b), int(act), L.ptr(out), n, D, H, W, C, L.stream())
    return out


def act_to_ncdhw(x: torch.Tensor) -> torch.Tensor:
    n, D, H, W, C = x.shape
    out = torch.empty(n, C, D, H, W, dtype=torch.float32, device=x.device)
    L.call("nm_ndhwc_to_ncdhw_f32", L.ptr(x), L.ptr(out), n, D * H * W, C, D * H * W * C, L.stream())
    return out


def ncdhw_to_act(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    x = x.float().contiguous()
    n, C, D, H, W = x.shape
    out = torch.empty(n, D, H, W, C, dtype=ACT_DTYPE, device=x.device)
    L.call("nm_ncdhw_f32_to_ndhwc", L.ptr(x), L.ptr(out), n, D * H * W, C, L.stream())
    return out


def mean_over_frames(seq: torch.Tensor) -> torch.Tensor:
    """(B, T, 1, G, G, G) fp32 -> (B, G, G, G)."""
    B, T = seq.shape[:2]
    G = seq.shape[-1]
    out = torch.empty(B, G, G, G, dtype=torch.float32, device=seq.device)
    L.call("nm_mean_over_frames", L.ptr(seq), L.ptr(out), B, T, G ** 3, L.stream())
    return out


def final_recon(raw, a, b, conv: torch.nn.Conv3d, first_frame, frames_per_clip, sharpness, translation,
                target=None, out=None, bce_out=None):
    """-> recon (n, G, G, G) fp32 [, per-frame BCE mean (n)]; `out` / `bce_out`: preallocated dense views."""
    n, D, H, W, C = raw.shape
    S = D * H * W
    recon = out if out is not None else torch.empty(n, D, H, W, dtype=torch.float32, device=raw.device)
    w = f32(conv, "weight").reshape(-1)
    bias_dev = f32(conv, "bias")                       # the live parameter, read on the device (no host sync per step)
    bce = None
    if target is not None:
        bce = bce_out if bce_out is not None else torch.empty(n, dtype=torch.float32, device=raw.device)
    ws = workspace(L.query("nm_final_recon_workspace_bytes", n), raw.device, "recon") if target is not None else None
    L.call("nm_final_recon", L.ptr(raw), L.ptr(a), L.ptr(b), L.ptr(w), 0.0, L.ptr(bias_dev), L.ptr(first_frame), frames_per_clip,
           float(sharpness), float(translation), L.ptr(recon), L.ptr(target), L.ptr(bce), L.ptr(ws), n, S, C,
           L.stream())
    return recon, bce


def chamfer_vol_fit(seq_frames: torch.Tensor, keypoints: torch.Tensor) -> torch.Tensor:
    """seq_frames (n, G, G, G) fp32, keypoints (n, K, 4) -> (n) fp32."""
    n, G = seq_frames.shape[0], seq_frames.shape[-1]
    K = keypoints.shape[1]
    out = torch.empty(n, dtype=torch.float32, device=seq_frames.device)
    ws = workspace(L.query("nm_chamfer_workspace_bytes", n), seq_frames.device, "chamfer")
    L.call("nm_chamfer_vol_fit", L.ptr(seq_frames), L.ptr(keypoints), L.ptr(linspace(G, seq_frames.device)), n, K, G,
           L.ptr(out), L.ptr(ws), L.stream())
    return out


# ------------------------------------------------------------------ heads
def _prop_dev(prop: torch.nn.Conv3d) -> torch.Tensor:
    """(w0, w1, bias) of the propagate conv (1, 2, 1, 1, 1) packed on the device: the kernels read it there, so a training
    loop never reads the updated parameters back to the host (that was two synchronisations in the middle of every step)."""
    return _cached(prop, "dev3", [prop.weight, prop.bias],
                   lambda: torch.cat([prop.weight.detach().float().reshape(-1), prop.bias.detach().float().reshape(-1)]).contiguous())


def heatmap_head(feature, conv1: torch.nn.Conv3d, K: int, mode: int, prev=None, frames_per_clip: int = 1,
                 prop: Optional[torch.nn.Conv3d] = None, sigma: float = 1.0, want_gaussians: bool = True,
                 out=None):
    """feature act (n, g, g, g, C).  mode 0 -> heat (n, K, g, g, g).
    mode 1 -> (heat, keypoints (n, K, 4), gaussians (n, K, g, g, g) | None, heat_mean (n, K)).
    `out` = preallocated dense (heat, keypoints, gaussians | None, heat_mean) views to write into."""
    n, g, C = feature.shape[0], feature.shape[1], feature.shape[-1]
    dev = feature.device
    heat = out[0] if out is not None else torch.empty(n, K, g, g, g, dtype=torch.float32, device=dev)
    w1 = f32(conv1, "weight").reshape(K, C)
    b1 = f32(conv1, "bias")
    if mode == 0:
        L.call("nm_heatmap_head", L.ptr(feature), L.ptr(w1), L.ptr(b1), n, g, C, K, 0, None, 1, 0.0, 0.0, 0.0, None,
               L.ptr(linspace(g, dev)), 1.0, L.ptr(heat), None, None, None, L.stream())
        return heat
    prop_dev = _prop_dev(prop)
    if out is not None:
        kp, gs, hm_mean = out[1], out[2], out[3]
    else:
        kp = torch.empty(n, K, 4, dtype=torch.float32, device=dev)
        gs = torch.empty(n, K, g, g, g, dtype=torch.float32, device=dev) if want_gaussians else None
        hm_mean = torch.empty(n, K, dtype=torch.float32, device=dev)
    L.call("nm_heatmap_head", L.ptr(feature), L.ptr(w1), L.ptr(b1), n, g, C, K, 1, L.ptr(prev), frames_per_clip,
           0.0, 0.0, 0.0, L.ptr(prop_dev), L.ptr(linspace(g, dev)), gauss_width(sigma, g), L.ptr(heat), L.ptr(kp), L.ptr(gs),
           L.ptr(hm_mean), L.stream())
    return heat, kp, gs, hm_mean


def gaussian_render(keypoints: torch.Tensor, sigma: float, g: int) -> torch.Tensor:
    """keypoints (n, K, 4) -> (n, K, g, g, g) fp32 (kypt_detector_utils.py:57-90, all keypoints at once)."""
    _need_cuda(keypoints)
    keypoints = keypoints.float().contiguous()
    n, K = keypoints.shape[:2]
    out = torch.empty(n, K, g, g, g, dtype=torch.float32, device=keypoints.device)
    L.call("nm_gaussian_render", L.ptr(keypoints), n, K, g, L.ptr(linspace(g, keypoints.device)),
           gauss_width(sigma, g), L.ptr(out), L.stream())
    return out


def decoder_adjust(ff_act, conv: torch.nn.Conv3d, frames_per_clip: int, g: int, K: int, sigma: float,
                   keypoints=None, gaussians=None) -> torch.Tensor:
    """ff_act (B, g, g, g, 128) act; keypoints (B*T, K, 4) or gaussians (B*T, K, g, g, g) -> act (B*T, g, g, g, 128)."""
    B = ff_act.shape[0]
    n = B * frames_per_clip
    dev = ff_act.device
    out = torch.empty(n, g, g, g, conv.out_channels, dtype=ACT_DTYPE, device=dev)
    assert conv.out_channels == 128 and conv.in_channels == 128 + 2 * K + 3
    base = workspace(L.query("nm_decoder_adjust_workspace_bytes", B, g), dev, "adjust")
    w = f32(conv, "weight").reshape(conv.out_channels, -1)
    L.call("nm_decoder_adjust", L.ptr(ff_act), L.ptr(keypoints), L.ptr(gaussians), L.ptr(w), L.ptr(f32(conv, "bias")),
           B, frames_per_clip, g, K, L.ptr(linspace(g, dev)), gauss_width(sigma, g), L.ptr(base), L.ptr(out),
           L.stream())
    return out


# ------------------------------------------------------------------ dynamics
def _hsvrnn_layers(mod):
    return [("post0", mod.extract_post_dist[0]), ("post2", mod.extract_post_dist[2]),
            ("prior0", mod.extract_prior_dist[0]), ("prior2", mod.extract_prior_dist[2]),
            ("root0", mod.root_intensity_decoder[0]), ("root2", mod.root_intensity_decoder[2]),
            ("joint0", mod.joint_matrix_decoder[0]), ("joint2", mod.joint_matrix_decoder[2])]


def hsvrnn_params(mod):
    """The parameters `nm_hsvrnn_weight_grads` differentiates, in the order of `L.HsvrnnGrads`."""
    cell = mod.kypt_rnn_cell
    return [p for _, lin in _hsvrnn_layers(mod) for p in (lin.weight, lin.bias)] + \
           [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh, mod.init_kypt_rnn_state, mod.offset_param]


def hsvrnn_weight_struct(mod, transposed: bool = True) -> "L.HsvrnnWeights":
    """The ctypes struct of the HSVRNN matrices: transposed fp32 copies ([in][out], what the step kernels read) or, with
    transposed=False, the fp32 parameters in their own [out][in] layout (what the backward's W^T dy products read)."""
    names = _hsvrnn_layers(mod)
    cell = mod.kypt_rnn_cell
    params = hsvrnn_params(mod)[:20]

    def build():
        keep = []
        st = L.HsvrnnWeights()
        f = (lambda p: p.detach().float().t().contiguous()) if transposed else (lambda p: p.detach().float().contiguous())
        for tag, lin in names:
            wt = f(lin.weight)
            b = lin.bias.detach().float().contiguous()
            keep += [wt, b]
            setattr(st, tag + "_wt", wt.data_ptr())
            setattr(st, tag + "_b", b.data_ptr())
        for tag, p in (("gru_ih_wt", cell.weight_ih), ("gru_hh_wt", cell.weight_hh)):
            wt = f(p)
            keep.append(wt)
            setattr(st, tag, wt.data_ptr())
        for tag, p in (("gru_ih_b", cell.bias_ih), ("gru_hh_b", cell.bias_hh)):
            b = p.detach().float().contiguous()
            keep.append(b)
            setattr(st, tag, b.data_ptr())
        return st, keep
    return _cached(mod, "hsvrnn" if transposed else "hsvrnn_oi", params, build)[0]


def hsvrnn_step(wstruct, h, kp_flat, eps, offset, order, parents, K: int, posterior: bool,
                want_z=False, want_R=False, want_post=False, want_prior=False):
    """One fused time step.  eps: (S, B, Z) for posterior steps, (B, Z) for prior steps."""
    B = h.shape[0]
    dev = h.device
    S = eps.shape[0] if posterior else 1
    h_out = torch.empty_like(h)
    kp_out = torch.empty(B, 4 * K, dtype=torch.float32, device=dev)
    z_out = torch.empty(B, eps.shape[-1], dtype=torch.float32, device=dev) if want_z else None
    R_out = torch.empty(B, K, 3, 3, dtype=torch.float32, device=dev) if want_R else None
    post = torch.empty(B, 2 * eps.shape[-1], dtype=torch.float32, device=dev) if want_post else None
    prior = torch.empty(B, 2 * eps.shape[-1], dtype=torch.float32, device=dev) if want_prior else None
    L.call("nm_hsvrnn_step", ctypes.byref(wstruct), L.ptr(h), L.ptr(kp_flat), L.ptr(eps), L.ptr(offset), L.ptr(order),
           L.ptr(parents), B, K, S, int(posterior), L.ptr(h_out), L.ptr(kp_out), L.ptr(z_out), L.ptr(R_out),
           L.ptr(post), L.ptr(prior), L.stream())
    return h_out, kp_out, z_out, R_out, post, prior


def hsvrnn_step_record(wstruct, h, kp_flat, eps, offset, order, parents, K: int, h_out, kp_out, z_out, R_out, post_out,
                       prior_out, pick_out):
    """A posterior `hsvrnn_step` into caller-provided outputs that also records the picked sample (pick_out (B) int32)."""
    _need_cuda(h, kp_flat, eps, offset, h_out, pick_out)
    L.call("nm_hsvrnn_step_record", ctypes.byref(wstruct), L.ptr(h), L.ptr(kp_flat), L.ptr(eps), L.ptr(offset),
           L.ptr(order), L.ptr(parents), h.shape[0], K, eps.shape[0], 1, L.ptr(h_out), L.ptr(kp_out), L.ptr(z_out),
           L.ptr(R_out), L.ptr(post_out), L.ptr(prior_out), L.ptr(pick_out), L.stream())


def hsvrnn_backward_workspace(B: int, T: int, device) -> torch.Tensor:
    """(T, B, row) fp32 records of the reverse loop; step t writes slice t."""
    row = L.query("nm_hsvrnn_backward_workspace_bytes", 1, 1) // 4
    return torch.empty(T, B, row, dtype=torch.float32, device=device)


def hsvrnn_step_backward(wt, w, h, kp_flat, eps, pick, f, z, R, offset, order, parents, K: int, dh_next, dh_ext, df, dR, dz,
                         dpost, dprior, dh_out, doffset, rows):
    """Backward of one conditioned step (see include/nm_b200.h): writes dh_out, accumulates doffset, fills rows."""
    _need_cuda(h, kp_flat, eps, pick, f, z, R, offset, dh_next, dh_ext, df, dR, dz, dpost, dprior, dh_out, doffset, rows)
    L.call("nm_hsvrnn_step_backward", ctypes.byref(wt), ctypes.byref(w), L.ptr(h), L.ptr(kp_flat), L.ptr(eps), L.ptr(pick),
           L.ptr(f), L.ptr(z), L.ptr(R), L.ptr(offset), L.ptr(order), L.ptr(parents), h.shape[0], K, eps.shape[0],
           L.ptr(dh_next), L.ptr(dh_ext), L.ptr(df), L.ptr(dR), L.ptr(dz), L.ptr(dpost), L.ptr(dprior), L.ptr(dh_out),
           L.ptr(doffset), L.ptr(rows), L.stream())


def hsvrnn_weight_grads(rows, h, kp, f, z, dh0, offset, doffset, offset_param, grads):
    """Every parameter gradient of the reverse loop in one launch.  grads: tensors shaped like `hsvrnn_params` (the last,
    offset_param's, may be None); all are fully overwritten."""
    _need_cuda(rows, h, kp, f, z, dh0, offset, doffset, offset_param)
    T, B = rows.shape[:2]
    K = kp.shape[-1] // 4
    g = L.HsvrnnGrads()
    for (name, _), t in zip(L.HsvrnnGrads._fields_, grads):
        _need_cuda(t)
        setattr(g, name, L.ptr(t))
    L.call("nm_hsvrnn_weight_grads", L.ptr(rows), L.ptr(h), L.ptr(kp), L.ptr(f), L.ptr(z), L.ptr(dh0), L.ptr(offset),
           L.ptr(doffset), L.ptr(offset_param), B, T, K, ctypes.byref(g), L.stream())


def hsvrnn_decode_pose(wstruct, dec_in, offset, order, parents, K: int):
    B = dec_in.shape[0]
    flat = torch.empty(B, 4 * K, dtype=torch.float32, device=dec_in.device)
    R = torch.empty(B, K, 3, 3, dtype=torch.float32, device=dec_in.device)
    L.call("nm_hsvrnn_decode_pose", ctypes.byref(wstruct), L.ptr(dec_in), L.ptr(offset), L.ptr(order), L.ptr(parents),
           B, K, L.ptr(flat), L.ptr(R), L.stream())
    return flat, R


def hsvrnn_bone_offsets(keypoints, parents, offset_param) -> torch.Tensor:
    B, T, K = keypoints.shape[:3]
    out = torch.empty(B, K, 3, dtype=torch.float32, device=keypoints.device)
    L.call("nm_hsvrnn_bone_offsets", L.ptr(keypoints), L.ptr(parents), L.ptr(offset_param), B, T, K, L.ptr(out),
           L.stream())
    return out


# ------------------------------------------------------------------ consumers of the path's outputs (SURVEY §8f#4)
def voxel_chamfer(gt: torch.Tensor, recon: torch.Tensor, binarize: bool = True, frames_per_call: int = 256):
    """gt, recon (n, G, G, G) fp32 dense -> (chamfer (n) fp32, occupied (n, 2) int32, err int32 scalar tensor).
    `recon` is binarised in place when `binarize` (utils/eval_utils.py:37-38)."""
    _need_cuda(gt)
    n, G = gt.shape[0], gt.shape[-1]
    out = torch.empty(n, dtype=torch.float32, device=gt.device)
    occ = torch.empty(n, 2, dtype=torch.int32, device=gt.device)
    err = torch.zeros(1, dtype=torch.int32, device=gt.device)
    step = max(1, min(frames_per_call, 65535))
    ws = workspace(L.query("nm_voxel_chamfer_workspace_bytes", min(n, step), G), gt.device, "voxel_chamfer")
    for s in range(0, n, step):
        m = min(step, n - s)
        L.call("nm_voxel_chamfer", L.ptr(gt[s:s + m]), L.ptr(recon[s:s + m]), m, G, int(binarize), L.ptr(out[s:s + m]),
               L.ptr(occ[s:s + m]), L.ptr(err), L.ptr(ws), L.stream())
    return out, occ, err


def semantic_nearest(keypoints: torch.Tensor, gt_keypoints: torch.Tensor, threshold: float = 0.2):
    """keypoints (F, K, 4) fp32 (masked in place), gt_keypoints (F, Kgt, 3) -> (idx (F, Kgt) int64, hist (Kgt, K) int32)."""
    _need_cuda(keypoints)
    F, K = keypoints.shape[0], keypoints.shape[1]
    Kgt = gt_keypoints.shape[1]
    idx = torch.empty(F, Kgt, dtype=torch.int64, device=keypoints.device)
    hist = torch.empty(Kgt, K, dtype=torch.int32, device=keypoints.device)
    L.call("nm_semantic_nearest", L.ptr(keypoints), L.ptr(gt_keypoints), F, K, Kgt, float(threshold), L.ptr(idx),
           L.ptr(hist), L.stream())
    return idx, hist


def skin_weights(points: torch.Tensor, keypoints: torch.Tensor, parents: torch.Tensor, root: int, hardness: float,
                 threshold: float):
    """points (N, 3), keypoints (K, 4) fp32, parents (K) int32 -> (skin (N, K) fp32, nearest (N) int32, err)."""
    _need_cuda(points)
    N, K = points.shape[0], keypoints.shape[0]
    skin = torch.empty(N, K, dtype=torch.float32, device=points.device)
    near = torch.empty(N, dtype=torch.int32, device=points.device)
    err = torch.zeros(1, dtype=torch.int32, device=points.device)
    L.call("nm_skin_weights", L.ptr(points), N, L.ptr(keypoints), L.ptr(parents), K, int(root), float(hardness),
           float(threshold), L.ptr(skin), L.ptr(near), L.ptr(err), L.stream())
    return skin, near, err


def retarget_fk(R: torch.Tensor, offset: torch.Tensor, root_pos: torch.Tensor, order: torch.Tensor,
                parents: torch.Tensor, clip: bool = True) -> torch.Tensor:
    """R (T, K, 3, 3), offset (K, 3), root_pos (T, 3), order / parents (K) int32 -> (T, K, 3)."""
    _need_cuda(R)
    T, K = R.shape[0], R.shape[1]
    pos = torch.empty(T, K, 3, dtype=torch.float32, device=R.device)
    L.call("nm_retarget_fk", L.ptr(R), L.ptr(offset), L.ptr(root_pos), L.ptr(order), L.ptr(parents), T, K, int(clip),
           L.ptr(pos), L.stream())
    return pos


def linear_blend_skinning(points, joints, R_inv, T3x4, skin) -> torch.Tensor:
    """points (N, 3), joints (K, 3), R_inv (K, 3, 3) | None, T3x4 (T, K, 3, 4), skin (N, K) -> (T, N, 3)."""
    _need_cuda(points)
    N, (T, K) = points.shape[0], T3x4.shape[:2]
    out = torch.empty(T, N, 3, dtype=torch.float32, device=points.device)
    L.call("nm_linear_blend_skinning", L.ptr(points), N, L.ptr(joints), L.ptr(R_inv), L.ptr(T3x4), L.ptr(skin), T, K,
           L.ptr(out), L.stream())
    return out
