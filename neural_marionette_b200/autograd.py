"""torch.autograd.Function wrappers that put the detector's training step (config #4: fwd + bwd of
`KyptDetector.forward`, reference train.py:387-409) on the nm_b200 kernels.

One Function per fused stage of the training-mode forward; autograd only does the bookkeeping (saved tensors, fan-out
sums, routing of the parameter gradients).  Activations and their gradients are fp16 channels-last tensors; activation
gradients carry a loss scale (`ops.grad_scale()`), every fp32 gradient that leaves a Function (parameters, keypoints)
has it divided out again, so `param.grad` holds true values as with the reference.

  FirstConvGNAct     add_coord_channels + Conv3d(k5) + GroupNorm + LeakyReLU      vox_modules.py:8-19, kypt_detector.py:266
  ConvGNAct          Conv3d | ConvTranspose3d + GroupNorm [+ LeakyReLU] [+ skip]  vox_modules.py:8-75
  Head / HeadST      1x1 heads, propagate conv, Softplus, soft-argmax             kypt_detector.py:273-297,311-316,336-343
  Adjust             Gaussian render + adjust_combined_representation             kypt_detector.py:381,404-408
  Upsample2x         nn.Upsample(scale 2, trilinear)                              kypt_detector.py:427,441
  ConvGNFinalRecon   last 3x3x3 conv + GN + LReLU + 1x1 conv + sigmoid/tanh + BCE kypt_detector.py:450-457,410,91-92
  ChamferVolFit      get_volume_fitting_loss('chamfer')                           utils/kypt_detector_utils.py:141-157

and, for stage 2 (training the dynamics module, reference train.py:146-147), fp32 throughout with no loss scale:

  HSVRNNEncode       the conditioned roll-out of HSVRNNBVH.encode                 model/hsvrnn_bvh.py:67-156
"""
from __future__ import annotations

import math
import os

import torch

from . import ops


# log2 of the magnitude the largest entry gradient (dL/d pre-sigmoid map) is scaled to.  fp16 tops out at 2^16 and the
# GroupNorm backward multiplies by 1/sigma of the normalised tensors, so gradients can grow by 2^10 and more on the way
# down: the default scales the entry gradient to O(1).  The measured gradient error does not depend on the scale from
# 2^8 to 2^19 (profiles/r02_training.md), i.e. underflow is not what limits the accuracy.  `FusedAdam.step` lowers the
# head-room by 2^2 whenever a step overflowed (and skipped) and raises it again slowly - dynamic loss scaling.
GRAD_HEADROOM_LOG2 = int(os.environ.get("NM_GRAD_HEADROOM_LOG2", "0"))
_HEADROOM = [GRAD_HEADROOM_LOG2]


def headroom_log2() -> int:
    return _HEADROOM[0]


def adjust_headroom(delta: int) -> int:
    _HEADROOM[0] = max(-16, min(8, _HEADROOM[0] + int(delta)))
    return _HEADROOM[0]


def _c(t):
    return t if t.is_contiguous() else t.contiguous()


# The largest incoming loss gradient decides the loss scale.  Reading it is a device -> host round trip in the middle of
# the step (the host would stall until the whole forward has run and then trail the GPU through the backward); in a
# training loop it is the same number every step (loss weight / number of frames), so the value read asynchronously
# during the PREVIOUS backward of the same shape is used and the fresh one is only checked when it has arrived.
_GMAX = {}


def _entry_gradient_max(dbce: torch.Tensor) -> float:
    key = (dbce.device.index, dbce.numel())
    slot = _GMAX.get(key)
    if slot is None:
        slot = _GMAX[key] = dict(pinned=torch.zeros(1, dtype=torch.float32).pin_memory(), event=torch.cuda.Event(), value=None)
    if slot["value"] is not None and torch.cuda.is_current_stream_capturing():
        return slot["value"]                                   # graph capture: the loss scale is frozen into the graph
    if slot["value"] is not None and slot["event"].query():
        slot["value"] = float(slot["pinned"][0])              # last step's read-back has landed
    if slot["value"] is None:
        slot["value"] = float(dbce.abs().max().item())         # first call: synchronous
    slot["pinned"].copy_(dbce.abs().max().reshape(1), non_blocking=True)
    slot["event"].record()
    return slot["value"]


def _stats(sink):
    """(mean_rstd, xsum) of the single GroupNorm a Function's forward finalised, or () when the kernel did not emit them."""
    return tuple(sink[0]) if len(sink) == 1 else ()


class FirstConvGNAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, occ, w, b, gamma, beta, conv, gn):
        with ops.capture_gn_stats() as sink:
            raw, a, sh = ops.first_conv(occ, conv, gn)
        ctx.save_for_backward(occ, raw, *_stats(sink))
        ctx.mods = (conv, gn)
        return ops.affine_act(raw, a, sh, True)

    @staticmethod
    def backward(ctx, dy):
        occ, raw, *stats = ctx.saved_tensors
        conv, gn = ctx.mods
        inv = 1.0 / ops.grad_scale()
        draw, dg, db, dbias = ops.groupnorm_backward(raw, _c(dy), gn, leaky=True, out_scale=inv, stats=stats or None)
        dw = ops.first_conv_weight_grad(occ, draw, out_scale=inv)
        return None, dw, dbias, dg, db, None, None


class ConvGNAct(torch.autograd.Function):
    """out = [LeakyReLU](GroupNorm(conv(x))) [+ res]; conv: nn.Conv3d (k1 / k3 stride 1, k2 stride 2) or
    nn.ConvTranspose3d(k2, s2)."""

    @staticmethod
    def forward(ctx, x, w, b, gamma, beta, res, conv, gn, act):
        transposed = isinstance(conv, torch.nn.ConvTranspose3d)
        with ops.capture_gn_stats() as sink:
            raw, a, sh = (ops.conv_transpose3d if transposed else ops.conv3d)(x, conv, gn)
        ctx.save_for_backward(x, raw, *_stats(sink))
        ctx.cfg = (conv, gn, bool(act), transposed, res is not None)
        return ops.affine_act(raw, a, sh, bool(act), x2=res)

    @staticmethod
    def backward(ctx, dy):
        x, raw, *stats = ctx.saved_tensors
        conv, gn, act, transposed, has_res = ctx.cfg
        dy = _c(dy)
        inv = 1.0 / ops.grad_scale()
        draw, dg, db, dbias = ops.groupnorm_backward(raw, dy, gn, leaky=act, out_scale=inv, stats=stats or None)
        if transposed:
            dw = ops.conv_transpose3d_weight_grad(x, draw, out_scale=inv)
            dx = ops.conv_transpose3d_input_grad(draw, conv) if ctx.needs_input_grad[0] else None
        else:
            dw = ops.conv3d_weight_grad(x, draw, k=conv.kernel_size[0], stride=conv.stride[0], out_scale=inv)
            dx = ops.conv3d_input_grad(draw, conv) if ctx.needs_input_grad[0] else None
        return dx, dw, dbias, dg, db, (dy if has_res else None), None, None, None


class Upsample2x(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return ops.upsample2x(x)

    @staticmethod
    def backward(ctx, dy):
        return ops.upsample2x_backward(_c(dy))


class HeadST(torch.autograd.Function):
    """prev = LeakyReLU(conv1x1(st_feature)) (B, K, g, g, g) fp32.  `link` is shared with `Head`: its backward leaves
    the per-frame gradient of the pre-Softplus maps there, and this backward sums it over the clip's frames inside the
    kernel (the gradient tensor autograd hands over is a placeholder then)."""

    @staticmethod
    def forward(ctx, feat, w, b, conv, K, link):
        ctx.save_for_backward(feat)
        ctx.cfg = (conv, K, link)
        return ops.heatmap_head(feat, conv, K, mode=0)

    @staticmethod
    def backward(ctx, dprev):
        (feat,) = ctx.saved_tensors
        conv, K, link = ctx.cfg
        dq = link.pop("dq", None)
        if dq is not None:
            dfeat, _, dw, db, _ = ops.heatmap_head_backward(feat, conv, K, 0, ops.grad_scale(), frames_per_clip=link["T"],
                                                            prop=link["prop"], dq_in=dq)
        else:
            dfeat, _, dw, db, _ = ops.heatmap_head_backward(feat, conv, K, 0, ops.grad_scale(), grad_heat=_c(dprev.float()))
        return dfeat, dw, db, None, None, None


class Head(torch.autograd.Function):
    """Per-frame heads: (heat (n, K, g, g, g), keypoints (n, K, 4), heat_mean (n, K)) from the feature map and the
    once-per-clip spatio-temporal heat-map `prev`."""

    @staticmethod
    def forward(ctx, feat, w1, b1, prev, pw, pb, conv1, prop, K, T, sigma, link):
        heat, kp, _, hmean = ops.heatmap_head(feat, conv1, K, mode=1, prev=prev, frames_per_clip=T, prop=prop, sigma=sigma,
                                              want_gaussians=False)
        ctx.save_for_backward(feat, prev, heat, kp, hmean)
        ctx.cfg = (conv1, prop, K, T, link)
        ctx.set_materialize_grads(False)
        return heat, kp, hmean

    @staticmethod
    def backward(ctx, dheat, dkp, dhmean):
        feat, prev, heat, kp, hmean = ctx.saved_tensors
        conv1, prop, K, T, link = ctx.cfg
        f = lambda t: None if t is None else _c(t.float())   # noqa: E731
        dfeat, dq, dw1, db1, dprop = ops.heatmap_head_backward(
            feat, conv1, K, 1, ops.grad_scale(), prev=prev, frames_per_clip=T, prop=prop, heat=heat, keypoints=kp,
            heat_mean=hmean, grad_keypoints=f(dkp), grad_heat_mean=f(dhmean), grad_heat=f(dheat))
        link.update(dq=dq, T=T, prop=prop)
        dprev = torch.zeros((), dtype=prev.dtype, device=prev.device).expand(prev.shape) if ctx.needs_input_grad[3] else None
        return dfeat, dw1, db1, dprev, dprop[:2].reshape(1, 2, 1, 1, 1), dprop[2:3], None, None, None, None, None, None


class Adjust(torch.autograd.Function):
    """act (B*T, g, g, g, 128) = LeakyReLU(adjust conv over cat[gauss_t, first_feature, gauss_0, coords])."""

    @staticmethod
    def forward(ctx, ff_act, kp, w, b, conv, T, g, K, sigma):
        y = ops.decoder_adjust(ff_act, conv, T, g, K, sigma, keypoints=kp)
        ctx.save_for_backward(ff_act, kp, y)
        ctx.cfg = (conv, T, g, K, sigma)
        return y

    @staticmethod
    def backward(ctx, dy):
        ff_act, kp, y = ctx.saved_tensors
        conv, T, g, K, sigma = ctx.cfg
        dff, dkp, dw, db = ops.decoder_adjust_backward(_c(dy), y, ff_act, kp, conv, T, g, K, sigma, ops.grad_scale())
        return dff, dkp, dw, db, None, None, None, None, None


class ConvGNFinalRecon(torch.autograd.Function):
    """(recon (n, G, G, G), per-frame BCE (n)) from the input of the decoder's last 3x3x3 conv.  Its backward is the
    first node of a backward pass through the reconstruction loss: it fixes the loss scale of that pass."""

    @staticmethod
    def forward(ctx, x, w11, b11, gamma, beta, w14, b14, first_frame, target, conv11, gn, conv14, T, sharp, trans):
        with ops.capture_gn_stats() as sink:
            raw, a, sh = ops.conv3d(x, conv11, gn)
        recon, bce = ops.final_recon(raw, a, sh, conv14, first_frame, T, sharp, trans, target=target)
        ctx.save_for_backward(x, raw, a, sh, recon, first_frame, target, *_stats(sink))
        ctx.cfg = (conv11, gn, conv14, T, sharp, trans)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(recon)
        return recon, bce

    @staticmethod
    def backward(ctx, _drecon, dbce):
        x, raw, a, sh, recon, first_frame, target, *stats = ctx.saved_tensors
        conv11, gn, conv14, T, sharp, trans = ctx.cfg
        if dbce is None:
            return (None,) * 15
        dbce = _c(dbce.float())
        S = raw.shape[1] * raw.shape[2] * raw.shape[3]
        # |dL/dx14| <= gmax * sharp / S; scale it to 2^headroom in fp16 (a power of two: exact scaling)
        gmax = _entry_gradient_max(dbce)
        if gmax > 0.0 and math.isfinite(gmax):
            ops.set_grad_scale(2.0 ** max(0, min(30, round(math.log2(S / (gmax * sharp))) + _HEADROOM[0])))
        scale = ops.grad_scale()
        if stats:
            # the tail's rank-one gradient is never materialised: dx14 per voxel + the GroupNorm-backward sums in one pass
            draw, dw14, db14, dg, db, dbias = ops.final_recon_backward_fused(raw, a, sh, conv14, gn, stats, sharp, recon, target,
                                                                           dbce, scale)
        else:
            dact, dw14, db14 = ops.final_recon_backward(raw, a, sh, conv14, first_frame, T, sharp, trans, recon, target, dbce,
                                                        scale)
            draw, dg, db, dbias = ops.groupnorm_backward(raw, dact, gn, leaky=True, out_scale=1.0 / scale)
        dw11 = ops.conv3d_weight_grad(x, draw, k=3, stride=1, out_scale=1.0 / scale)
        dx = ops.conv3d_input_grad(draw, conv11) if ctx.needs_input_grad[0] else None
        return (dx, dw11, dbias, dg, db, dw14, db14) + (None,) * 8


class ChamferVolFit(torch.autograd.Function):
    @staticmethod
    def forward(ctx, frames, kp):
        ctx.save_for_backward(frames, kp)
        return ops.chamfer_vol_fit(frames, kp)

    @staticmethod
    def backward(ctx, dout):
        frames, kp = ctx.saved_tensors
        return None, ops.chamfer_vol_fit_backward(frames, kp, _c(dout.float()))


class HSVRNNEncode(torch.autograd.Function):
    """The T recorded steps of `HSVRNNBVH.encode` (the eval loop, plus the pick of every element) -> per-step tensors
    f (B, T, K, 4), R (B, T, K, 3, 3), z (B, T, Z), h (B, T+1, H), post / prior (T, B, 2Z) = mean | std.  The backward
    runs `nm_hsvrnn_step_backward` from t = T-1 down to 0, then `nm_hsvrnn_weight_grads` once.  `params` are
    `ops.hsvrnn_params(mod)`, so autograd routes their gradients into `param.grad`; keypoints get none."""

    @staticmethod
    def forward(ctx, kp, eps, mod, *params):
        B, T, K, _ = kp.shape
        S, Z, H = eps.shape[1], mod.nlatent_kypt, mod.nhidden_kypt
        dev = kp.device
        order, parents = mod._tree(dev)
        w = ops.hsvrnn_weight_struct(mod)
        offset = ops.hsvrnn_bone_offsets(kp, parents, ops.f32(mod, "offset_param"))
        kpt = kp.transpose(0, 1).reshape(T, B, 4 * K).contiguous()
        hs = torch.empty(T + 1, B, H, dtype=torch.float32, device=dev)
        hs[0] = mod.init_kypt_rnn_state.detach().float().expand(B, -1)
        fs = torch.empty(T, B, 4 * K, dtype=torch.float32, device=dev)
        zs = torch.empty(T, B, Z, dtype=torch.float32, device=dev)
        Rs = torch.empty(T, B, K, 3, 3, dtype=torch.float32, device=dev)
        post = torch.empty(T, B, 2 * Z, dtype=torch.float32, device=dev)
        prior = torch.empty(T, B, 2 * Z, dtype=torch.float32, device=dev)
        pick = torch.empty(T, B, dtype=torch.int32, device=dev)
        for t in range(T):
            ops.hsvrnn_step_record(w, hs[t], kpt[t], eps[t], offset, order, parents, K, hs[t + 1], fs[t], zs[t], Rs[t],
                                   post[t], prior[t], pick[t])
        ctx.save_for_backward(hs, kpt, fs, zs, Rs, eps, pick, offset)
        ctx.mod = mod
        return (fs.view(T, B, K, 4).transpose(0, 1).contiguous(), Rs.transpose(0, 1).contiguous(),
                zs.transpose(0, 1).contiguous(), hs.transpose(0, 1).contiguous(), post, prior)

    @staticmethod
    def backward(ctx, dF, dR, dZ, dH, dpost, dprior):
        hs, kpt, fs, zs, Rs, eps, pick, offset = ctx.saved_tensors
        mod = ctx.mod
        T, B = fs.shape[:2]
        K = fs.shape[-1] // 4
        order, parents = mod._tree(hs.device)
        wt, w = ops.hsvrnn_weight_struct(mod), ops.hsvrnn_weight_struct(mod, transposed=False)
        dF = dF.float().transpose(0, 1).reshape(T, B, 4 * K).contiguous()
        dR = dR.float().transpose(0, 1).reshape(T, B, K * 9).contiguous()
        dZ = dZ.float().transpose(0, 1).contiguous()
        dH = dH.float().transpose(0, 1).contiguous()
        dpost, dprior = _c(dpost.float()), _c(dprior.float())
        rows = ops.hsvrnn_backward_workspace(B, T, hs.device)
        doff = torch.zeros_like(offset)
        carry, nxt = dH[T].clone(), torch.empty_like(dH[T])
        for t in range(T - 1, -1, -1):
            ops.hsvrnn_step_backward(wt, w, hs[t], kpt[t], eps[t], pick[t], fs[t], zs[t], Rs[t], offset, order, parents, K,
                                     carry, dH[t], dF[t], dR[t], dZ[t], dpost[t], dprior[t], nxt, doff, rows[t])
            carry, nxt = nxt, carry
        params = ops.hsvrnn_params(mod)
        want_op = ctx.needs_input_grad[3 + len(params) - 1]
        grads = [torch.empty(p.shape, dtype=torch.float32, device=p.device) for p in params[:-1]]
        grads.append(torch.empty(params[-1].shape, dtype=torch.float32, device=hs.device) if want_op else None)
        ops.hsvrnn_weight_grads(rows, hs, kpt, fs, zs, carry, offset, doff,
                                ops.f32(mod, "offset_param") if want_op else None, grads)
        return (None, None, None) + tuple(g if need else None for g, need in zip(grads, ctx.needs_input_grad[3:]))


# ------------------------------------------------------------------ module-level helpers used by the training path
def conv_gn_act(x, conv, gn, act=True, res=None):
    return ConvGNAct.apply(x, conv.weight, conv.bias, gn.weight, gn.bias, res, conv, gn, act)


def first_conv_gn_act(occ, conv, gn):
    return FirstConvGNAct.apply(occ, conv.weight, conv.bias, gn.weight, gn.bias, conv, gn)
