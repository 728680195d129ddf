"""HSVRNN latent dynamics over a learned skeleton (drop-in for the reference's model/hsvrnn_bvh.py).

Same class / parameter / attribute names (`extract_post_dist`, `extract_prior_dist`,
`root_intensity_decoder`, `joint_matrix_decoder`, `kypt_rnn_cell`, `init_kypt_rnn_state`, `offset_param`,
`A`, `priority`, `parents`) because the reference's demo scripts reach inside the module.  `encode` /
`generate` run ONE fused CUDA kernel per time step (`nm_hsvrnn_step`) instead of ~4.7k ATen launches.  In training mode
with autograd on, `encode` is differentiable (stage 2 of the reference's train.py): `autograd.HSVRNNEncode` runs the same
steps and backpropagates through time on the `nm_hsvrnn_step_backward` / `nm_hsvrnn_weight_grads` kernels.

Random draws: the reference calls `Normal.rsample`, i.e. standard-normal noise of shape (S, B, Z) per
conditioned step and (B, Z) per generated step, in time order.  The same draws are made here with
`torch.randn` on the module's device (or taken from the optional `eps*` arguments, which is how the parity
tests inject identical noise into both implementations).
"""
from __future__ import annotations

import torch
from torch import nn

from .. import ops
from ..autograd import HSVRNNEncode
from ..utils.dyna_utils import process_affinity_glob


def _mlp(n_in, n_out, tanh=False):
    layers = [nn.Linear(n_in, 128), nn.LeakyReLU(), nn.Linear(128, n_out)]
    if tanh:
        layers.append(nn.Tanh())
    return nn.Sequential(*layers)


class HSVRNNBVH(nn.Module):

    def __init__(self, options):
        super().__init__()
        self.nkeypoints = options.nkeypoints
        self.nlatent_kypt = options.nlatent_kypt
        self.nhidden_kypt = options.nhidden_kypt
        self.input_dim = options.input_dim
        self.transition_type = options.transition_type
        self.state_mode = options.state_mode
        self.action_mode = options.action_mode
        if self.transition_type != "dl" or self.input_dim != 3 or self.nhidden_kypt != 512 or self.nlatent_kypt != 128:
            raise NotImplementedError("only transition_type='dl', input_dim=3, nhidden_kypt=512, nlatent_kypt=128 "
                                      "(the shipped configuration) is implemented")
        if not 2 <= self.nkeypoints <= 64:
            raise NotImplementedError(f"nkeypoints={self.nkeypoints}: only 2 <= nkeypoints <= 64 is implemented "
                                      "(the CUDA kernels are compiled for at most 64 keypoints)")
        state_dim = self.nkeypoints * (self.input_dim + 1)
        H, Z = self.nhidden_kypt, self.nlatent_kypt
        self.extract_post_dist = _mlp(H + state_dim, 2 * Z)
        self.extract_prior_dist = _mlp(H, 2 * Z)
        self.root_intensity_decoder = _mlp(H + Z, 3 + self.nkeypoints, tanh=True)
        self.joint_matrix_decoder = _mlp(H + Z, 6 * self.nkeypoints)
        self.kypt_rnn_cell = nn.GRUCell(input_size=state_dim + Z, hidden_size=H)
        self.init_kypt_rnn_state = nn.Parameter(torch.randn(1, H))
        self.A, self.priority, self.parents = None, None, None
        self.offset_param = nn.Parameter(torch.randn(self.nkeypoints, 3))
        self.offset_param.requires_grad = False

    # ------------------------------------------------------------------ helpers
    def _tree(self, device):
        """int32 device copies of (priority.indices, parents) for the kernels."""
        key = (self.priority.indices.data_ptr(), self.parents.data_ptr(), str(device))
        cached = self.__dict__.get("_nm_tree")
        if cached is None or cached[0] != key:
            cached = (key, self.priority.indices.to(device=device, dtype=torch.int32).contiguous(),
                      self.parents.to(device=device, dtype=torch.int32).contiguous())
            self.__dict__["_nm_tree"] = cached
        return cached[1], cached[2]

    def _ensure_skeleton(self, affinity):
        if self.A is None:
            if affinity is None:
                raise ValueError("the skeleton is built from the affinity on the first encode() call")
            A, priority, parents = process_affinity_glob(affinity)
            self.A, self.priority, self.parents = A.float(), priority, parents

    def _guard(self):
        if self.training and torch.is_grad_enabled():
            raise NotImplementedError("neural_marionette_b200: HSVRNN backward kernels are not implemented yet; "
                                      "use .eval() / torch.no_grad()")

    def get_offset(self, keypoints):
        """(B, T, K, 4) -> (B, K, 3, 1): median parent distance x unit `offset_param` (reference :236-253)."""
        _, parents = self._tree(keypoints.device)
        with torch.no_grad():
            off = ops.hsvrnn_bone_offsets(keypoints.float().contiguous(), parents,
                                          ops.f32(self, "offset_param"))
        return off[..., None]

    def extract_kypt_from_latent_and_state(self, decoder_input, offset):
        """(B, 640), (B, K, 3, 1) -> (flat keypoints (B, 4K), global rotations (B, K, 3, 3)) (reference :255-286)."""
        order, parents = self._tree(decoder_input.device)
        B = decoder_input.shape[0]
        with torch.no_grad():
            off = offset.expand(B, self.nkeypoints, 3, 1).reshape(B, self.nkeypoints, 3).float().contiguous()
            return ops.hsvrnn_decode_pose(ops.hsvrnn_weight_struct(self), decoder_input.float().contiguous(), off,
                                          order, parents, self.nkeypoints)

    # ------------------------------------------------------------------ rollouts
    def encode(self, keypoints, affinity, SAMPLE_NUM=10, eps=None):
        """Track a keypoint sequence (reference :67-156).  keypoints (B, T, K, 4); eps optional (T, S, B, Z).
        Differentiable in training mode with grad enabled (the parameters only: keypoints must not require grad)."""
        if self.training and torch.is_grad_enabled():
            return self._encode_train(keypoints, affinity, SAMPLE_NUM, eps)
        B, T, K, _ = keypoints.shape
        dev = keypoints.device
        self._ensure_skeleton(affinity)
        order, parents = self._tree(dev)
        with torch.no_grad():
            kp = keypoints.float().contiguous()
            w = ops.hsvrnn_weight_struct(self)
            offset = ops.hsvrnn_bone_offsets(kp, parents, ops.f32(self, "offset_param"))
            h = self.init_kypt_rnn_state.detach().float().expand(B, -1).contiguous()
            hs, zs, kps, Rs, kls = [h], [], [], [], []
            Z = self.nlatent_kypt
            for t in range(T):
                e = eps[t] if eps is not None else torch.randn(SAMPLE_NUM, B, Z, device=dev)
                h, f, z, R, post, prior = ops.hsvrnn_step(w, h, kp[:, t].reshape(B, -1).contiguous(),
                                                          e.float().contiguous(), offset, order, parents, K, True,
                                                          want_z=True, want_R=True, want_post=True, want_prior=True)
                qm, qs, pm, ps = post[:, :Z], post[:, Z:], prior[:, :Z], prior[:, Z:]
                ratio = (qs / ps).pow(2)
                kls.append(0.5 * (ratio + ((qm - pm) / ps).pow(2) - 1 - ratio.log()))
                hs.append(h), zs.append(z), kps.append(f.view(B, K, 4)), Rs.append(R)
            inferred = torch.stack(kps, dim=1)
            return dict(
                kypt_recon=inferred[..., :4], R=torch.stack(Rs, dim=1), z_kypts=torch.stack(zs, dim=1),
                h_kypts=torch.stack(hs, dim=1), kl_kypt=torch.stack(kls, dim=1).mean(),
                kypt_recon_loss=(inferred - kp).pow(2).sum(dim=(2, 3)).mean(),
                gae_recon_loss=torch.tensor(0).to(dev), topo_recon_loss=torch.tensor(0).to(dev))

    def _encode_train(self, keypoints, affinity, SAMPLE_NUM, eps):
        if keypoints.requires_grad:
            raise NotImplementedError("neural_marionette_b200: HSVRNNBVH.encode has no gradient for the keypoints; pass "
                                      "keypoints.detach() (as NeuralMarionette.forward and the reference do)")
        B, T, K, _ = keypoints.shape
        dev = keypoints.device
        self._ensure_skeleton(affinity)
        Z = self.nlatent_kypt
        kp = keypoints.float().contiguous()
        if eps is None:     # the same draws, in the same order, as the step loop of the eval path
            eps = torch.stack([torch.randn(SAMPLE_NUM, B, Z, device=dev) for _ in range(T)])
        f, R, z, h, post, prior = HSVRNNEncode.apply(kp, eps.float().contiguous(), self, *ops.hsvrnn_params(self))
        kls = []
        for t in range(T):       # the eval path's expressions on the same (B, 2Z) slices: bit-identical values
            qm, qs, pm, ps = post[t][:, :Z], post[t][:, Z:], prior[t][:, :Z], prior[t][:, Z:]
            ratio = (qs / ps).pow(2)
            kls.append(0.5 * (ratio + ((qm - pm) / ps).pow(2) - 1 - ratio.log()))
        return dict(
            kypt_recon=f[..., :4], R=R, z_kypts=z, h_kypts=h, kl_kypt=torch.stack(kls, dim=1).mean(),
            kypt_recon_loss=(f - kp).pow(2).sum(dim=(2, 3)).mean(),      # zeros made on the device: no host copy
            gae_recon_loss=torch.zeros((), dtype=torch.int64, device=dev),
            topo_recon_loss=torch.zeros((), dtype=torch.int64, device=dev))

    def generate(self, keypoints_cond, affinity=None, Ttot=10, Tcond=3, SAMPLE_NUM=10, eps_cond=None, eps_gen=None):
        """Condition on Tcond detected frames, then roll the prior out to Ttot (reference :158-234).
        eps_cond optional (Tcond, S, B, Z); eps_gen optional (Ttot - Tcond, B, Z)."""
        self._guard()
        B, _, K, _ = keypoints_cond.shape
        dev = keypoints_cond.device
        if self.parents is None:
            raise TypeError("HSVRNNBVH.generate needs the skeleton: call encode() (or NeuralMarionette.forward) once "
                            "first, as the reference requires")
        order, parents = self._tree(dev)
        Z = self.nlatent_kypt
        with torch.no_grad():
            kp = keypoints_cond.float().contiguous()
            w = ops.hsvrnn_weight_struct(self)
            offset = ops.hsvrnn_bone_offsets(kp, parents, ops.f32(self, "offset_param"))
            h = self.init_kypt_rnn_state.detach().float().expand(B, -1).contiguous()
            cond, gen = [], []
            for t in range(Tcond):
                e = eps_cond[t] if eps_cond is not None else torch.randn(SAMPLE_NUM, B, Z, device=dev)
                h, f, *_ = ops.hsvrnn_step(w, h, kp[:, t].reshape(B, -1).contiguous(), e.float().contiguous(),
                                           offset, order, parents, K, True)
                cond.append(f.view(B, K, 4))
            for t in range(Tcond, Ttot):
                e = eps_gen[t - Tcond] if eps_gen is not None else torch.randn(B, Z, device=dev)
                h, f, *_ = ops.hsvrnn_step(w, h, None, e.float().contiguous(), offset, order, parents, K, False)
                gen.append(f.view(B, K, 4))
            return dict(keypoints_cond=torch.stack(cond, dim=1)[..., :4],
                        keypoints_gen=torch.stack(gen, dim=1)[..., :4])

    def interpolate(self, keypoints, affinity, sample_num=32, sample_rate=10, eps=None):
        """Key-frame interpolation with `sample_num` hypotheses — the loop the reference keeps inline in
        `vis_interpolation.py:86-136`, on the fused step kernels (one `nm_hsvrnn_step` per frame plus one
        `nm_hsvrnn_decode_pose` per key frame instead of ~40 module calls; no host sync inside the loop).
        keypoints (1, T, K, 4) detected on the clip; key frames are `t % sample_rate == 0` and the last frame.
        eps optional (T, 2, sample_num, Z): [t, 0] the posterior (key frame) / prior (in-between) draw, [t, 1] the
        prior draw "for choosing".  Returns dict(keypoints (1, T, K, 4) with the first frame's intensities,
        picks (n_key, 2) int64: surviving hypothesis / emitted hypothesis per key frame)."""
        self._guard()
        B, T, K, _ = keypoints.shape
        if B != 1:
            raise ValueError("interpolate works on one clip (the reference's loop expands it to sample_num hypotheses)")
        dev = keypoints.device
        self._ensure_skeleton(affinity)
        order, parents = self._tree(dev)
        Z, S = self.nlatent_kypt, int(sample_num)
        with torch.no_grad():
            kp = keypoints.float().contiguous()
            w = ops.hsvrnn_weight_struct(self)
            offset = ops.hsvrnn_bone_offsets(kp, parents, ops.f32(self, "offset_param")).expand(S, -1, -1).contiguous()
            h = self.init_kypt_rnn_state.detach().float().expand(S, -1).contiguous()
            selected, pending, picks = [], [], []
            for t in range(T):
                kp_flat = kp[:, t].reshape(1, -1).expand(S, -1).contiguous()
                e = eps[t].float() if eps is not None else torch.randn(2, S, Z, device=dev)
                if t % sample_rate == 0 or t == T - 1:
                    h_new, f, _, _, _, prior = ops.hsvrnn_step(w, h, kp_flat, e[0:1].contiguous(), offset, order, parents,
                                                               K, True, want_prior=True)
                    zc = prior[:, :Z] + prior[:, Z:] * e[1]
                    fc, _ = ops.hsvrnn_decode_pose(w, torch.cat([h, zc], dim=-1).contiguous(), offset, order, parents, K)
                    i = (f - kp_flat).pow(2).sum(dim=-1).argmin()
                    j = (fc - f[i][None]).pow(2).sum(dim=-1).argmin()
                    h = h_new[i][None].expand(S, -1).contiguous()      # GRU(cat[f_i, z_i], h_i) == the collapsed update
                    pending.append(kp_flat)
                    selected += [s[j].view(K, 4) for s in pending]
                    pending = []
                    picks.append(torch.stack([i, j]))
                else:
                    h, f, *_ = ops.hsvrnn_step(w, h, None, e[0].contiguous(), offset, order, parents, K, False)
                    pending.append(f)
            sel = torch.stack(selected, dim=0)[None].clone()
            sel[0, :, :, -1] = sel[0, 0, :, -1]
            return dict(keypoints=sel, picks=torch.stack(picks, dim=0))
