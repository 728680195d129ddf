"""Volumetric keypoint detector (drop-in for the reference's model/kypt_detector.py).

Same classes (`KyptDetector`, `VoxToKyptNet`, `KyptToVoxNet`), constructor arguments, sub-module / parameter
names and forward signatures as the reference, so `load_state_dict(strict=True)` accepts its checkpoints; the
arithmetic runs through the nm_b200 CUDA kernels:

  * all frames of all clips go through the feature net as ONE batch (frames are independent given the
    once-per-clip spatio-temporal heat-map) instead of the reference's Python loop over t;
  * the CoordConv channels are synthesised inside the first conv, GroupNorm is folded to per-sample
    scale/shift applied by the consumer, the heat-map head + soft-argmax + Gaussian render are one kernel,
    the decoder's 179-channel concat is never built (its clip-constant part is hoisted), the final 1x1 conv,
    tanh/sigmoid and the BCE reduction are one kernel.

Training (`net.train()` with autograd enabled, reference train.py:387-409): `KyptDetector.forward` runs the same
kernels through the autograd Functions of `neural_marionette_b200/autograd.py`; `loss.backward()` then runs the backward
kernels (data / weight gradients of the convs, GroupNorm, up-sampling, heads, render, losses) and leaves fp32 gradients
in `param.grad` like the reference.  `VoxToKyptNet.forward` / `KyptToVoxNet.forward` on their own stay inference-only.
"""
from __future__ import annotations

import torch
from torch import nn

from .. import autograd as AG
from .. import ops
from ..modules.vox_modules import HG, Basic3DBlock, Pool3DBlock, Res3DBlock
from ..utils.kypt_detector_utils import (get_graph_consistency_loss, get_graph_traj_loss,
                                         get_temporal_separation_loss, get_volume_fitting_loss,
                                         sparsity_loss_from_means)

# Frames pushed through the conv stack per pass.  Bounds activation memory (the widest tensors are 32 ch @ G^3 =
# 16.8 MB/frame at G = 64 -> ~11 GB each at 640 frames, ~45 GB live) while keeping every launch large: the hour-glass
# levels <= 8^3 are launch-latency bound, so bigger passes amortise them.  Measured on one B200 (B = 64, T = 20, same
# GPU): 320 frames/pass 168.5 ms/step, 640 -> 166.9, 1280 -> 166.3.
FRAME_CHUNK = int(__import__("os").environ.get("NM_FRAME_CHUNK", "640"))


def frames_per_pass(grid_size: int) -> int:
    """FRAME_CHUNK is quoted for grid 64^3; other grids keep the same activation footprint (G = 128: 80 frames)."""
    return max(1, FRAME_CHUNK * 64 ** 3 // grid_size ** 3)
# Run the once-per-clip spatio-temporal branch on an auxiliary stream next to the per-frame encoder (0 disables).
ST_OVERLAP = __import__("os").environ.get("NM_ST_OVERLAP", "1") != "0"
# Interpolate the first decoder up-sampling inside the dec.1 conv as well (0: separate up-sampling kernel).
UP_DEC1 = __import__("os").environ.get("NM_UP_DEC1", "1") != "0"


def _training(module) -> bool:
    return module.training and torch.is_grad_enabled()


def _no_training(module):
    if _training(module):
        raise NotImplementedError(
            "neural_marionette_b200: autograd is wired through KyptDetector.forward only; call this sub-module under "
            "torch.no_grad() / .eval(), or train through KyptDetector / NeuralMarionette")


def _heatmap_net(in_channels, out_channels, act):
    layer = nn.Softplus() if act == "softplus" else nn.LeakyReLU()
    return nn.Sequential(nn.Conv3d(in_channels, out_channels, kernel_size=1, stride=1, padding=0), layer)


def _feature_net(in_channels, out_channels, grid_size):
    return nn.Sequential(
        Basic3DBlock(1 + in_channels, out_channels // 4, 5),
        Pool3DBlock(2, out_channels // 4),
        Res3DBlock(out_channels // 4, out_channels // 2),
        Pool3DBlock(2, out_channels // 2),
        HG(out_channels // 2, out_channels // 2, N=grid_size // 4),
        Res3DBlock(out_channels // 2, out_channels))


def run_feature_net(net: nn.Sequential, occ: torch.Tensor) -> torch.Tensor:
    """occ (n, G, G, G) fp32 -> act (n, G/4, G/4, G/4, C)."""
    # the first layer's GroupNorm + LeakyReLU is applied inside the pool conv that follows
    raw, a, b = net[0].run_coordconv_raw(occ)
    x = net[1].run(raw, in_affine=(a, b, True))
    # the two normalised branches of the first Res3DBlock are summed inside the second pool conv
    raw, a, b, x2, a2, b2 = net[2].run_raw(x)
    x = net[3].run(raw, in_affine=(a, b, False, x2, a2, b2))
    for block in list(net)[4:]:
        x = block.run(x)
    return x


def run_feature_net_train(net: nn.Sequential, occ: torch.Tensor) -> torch.Tensor:
    """Training-mode feature net: every block through its autograd Function (activations kept for the backward)."""
    x = net[0].run_coordconv_train(occ)
    for block in list(net)[1:]:
        x = block.run_train(x)
    return x


class VoxToKyptNet(nn.Module):
    """Occupancy clips -> heat-maps, keypoints, Gaussian maps (reference kypt_detector.py:244-365)."""

    def __init__(self, grid_size, nkeypoints, input_dim, sigmas, fixed_sigma, const_intensity):
        super().__init__()
        if const_intensity != 3 or not fixed_sigma or input_dim != 3:
            raise NotImplementedError("only the shipped configuration (const_intensity=3, fixed_sigma=1, "
                                      "input_dim=3) is implemented")
        self.grid_size = grid_size
        self.feat_dim = 128
        self.nkeypoints = nkeypoints
        self.fixed_sigma = fixed_sigma
        self.const_intensity = const_intensity
        self.sigmas = sigmas
        self.extract_features = _feature_net(input_dim, self.feat_dim, grid_size)
        self.extract_heatmaps_from_features = _heatmap_net(self.feat_dim, nkeypoints, "leakyrelu")
        self.extract_spatio_temporal_features = _feature_net(input_dim, self.feat_dim * 2, grid_size)
        self.extract_spatio_temporal_heatmaps_from_features = _heatmap_net(self.feat_dim * 2, nkeypoints, "leakyrelu")
        self.propagate_heatmaps = nn.Sequential(nn.Conv3d(2, 1, kernel_size=1, stride=1, padding=0), nn.Softplus())

    def detect(self, seq, want_gaussians=True):
        """seq (B, T, 1, G, G, G) fp32 CUDA.  Returns dict(heatmaps, keypoints, gaussians, first_feature,
        first_feature_act, heat_mean)."""
        _no_training(self)
        B, T = seq.shape[:2]
        G, K, g = self.grid_size, self.nkeypoints, self.grid_size // 4
        assert seq.shape[2] == 1 and tuple(seq.shape[3:]) == (G, G, G), "expected (B, T, 1, G, G, G) occupancy"
        seq = seq.float().contiguous()
        sigma = float(self.sigmas[0])
        with torch.no_grad():
            # once per clip: spatio-temporal heat-map from the frame mean (never updated for const_intensity 3).
            # Its ~170 mostly small launches run on an auxiliary stream, next to the per-frame encoder of the first
            # pass; the per-frame head waits for it.
            main = torch.cuda.current_stream(seq.device)
            side = ops.side_stream(seq.device) if ST_OVERLAP else main
            if side is not main:
                side.wait_stream(main)
            with torch.cuda.stream(side):
                st = run_feature_net(self.extract_spatio_temporal_features, ops.mean_over_frames(seq))
                prev = ops.heatmap_head(st, self.extract_spatio_temporal_heatmaps_from_features[0], K, mode=0)
                del st
            if side is not main:
                prev.record_stream(main)
                seq.record_stream(side)
            st_pending = side is not main
            frames = seq.view(B * T, G, G, G)
            heat = torch.empty(B * T, K, g, g, g, dtype=torch.float32, device=seq.device)
            kps = torch.empty(B * T, K, 4, dtype=torch.float32, device=seq.device)
            gss = torch.empty(B * T, K, g, g, g, dtype=torch.float32, device=seq.device) if want_gaussians else None
            hmean = torch.empty(B * T, K, dtype=torch.float32, device=seq.device)
            ff_act = torch.empty(B, g, g, g, self.feat_dim, dtype=ops.ACT_DTYPE, device=seq.device)
            clips = max(1, frames_per_pass(G) // T)
            for b0 in range(0, B, clips):
                b1 = min(B, b0 + clips)
                feat = run_feature_net(self.extract_features, frames[b0 * T:b1 * T])
                ff_act[b0:b1] = feat.view(b1 - b0, T, g, g, g, self.feat_dim)[:, 0]
                sl = slice(b0 * T, b1 * T)
                if st_pending:
                    main.wait_stream(side)
                    st_pending = False
                ops.heatmap_head(feat, self.extract_heatmaps_from_features[0], K, mode=1, prev=prev[b0:b1],
                                 frames_per_clip=T, prop=self.propagate_heatmaps[0], sigma=sigma,
                                 want_gaussians=want_gaussians,
                                 out=(heat[sl], kps[sl], gss[sl] if want_gaussians else None, hmean[sl]))
            return dict(heatmaps=heat.view(B, T, K, g, g, g), keypoints=kps.view(B, T, K, 4),
                        gaussians=gss.view(B, T, K, g, g, g) if want_gaussians else None,
                        first_feature=ops.act_to_ncdhw(ff_act), first_feature_act=ff_act,
                        heat_mean=hmean.view(B, T, K))

    def detect_train(self, seq):
        """Training-mode `detect` (autograd): same outputs, `gaussians` omitted (the decoder re-renders them from the
        keypoints), `first_feature_act` / `keypoints` / `heat_mean` carry the graph."""
        B, T = seq.shape[:2]
        G, K, g = self.grid_size, self.nkeypoints, self.grid_size // 4
        assert seq.shape[2] == 1 and tuple(seq.shape[3:]) == (G, G, G), "expected (B, T, 1, G, G, G) occupancy"
        if B * T > frames_per_pass(G):
            raise ValueError(f"training step: {B * T} frames exceed one pass ({frames_per_pass(G)}); lower the batch "
                             "or raise NM_FRAME_CHUNK")
        seq = seq.detach().float().contiguous()
        sigma = float(self.sigmas[0])
        link = {}
        st = run_feature_net_train(self.extract_spatio_temporal_features, ops.mean_over_frames(seq))
        st_head = self.extract_spatio_temporal_heatmaps_from_features[0]
        prev = AG.HeadST.apply(st, st_head.weight, st_head.bias, st_head, K, link)
        feat = run_feature_net_train(self.extract_features, seq.view(B * T, G, G, G))
        head, prop = self.extract_heatmaps_from_features[0], self.propagate_heatmaps[0]
        heat, kps, hmean = AG.Head.apply(feat, head.weight, head.bias, prev, prop.weight, prop.bias, head, prop, K, T,
                                         sigma, link)
        ff_act = feat.view(B, T, g, g, g, self.feat_dim)[:, 0].contiguous()
        return dict(heatmaps=heat.view(B, T, K, g, g, g), keypoints=kps.view(B, T, K, 4), gaussians=None,
                    first_feature=ops.act_to_ncdhw(ff_act.detach()), first_feature_act=ff_act,
                    heat_mean=hmean.view(B, T, K))

    def forward(self, seq, Tcond=None):
        out = self.detect(seq)
        return out["heatmaps"], out["keypoints"], out["gaussians"], out["first_feature"]


class KyptToVoxNet(nn.Module):
    """Keypoint Gaussians + first-frame feature -> occupancy reconstruction (reference kypt_detector.py:369-460)."""

    def __init__(self, grid_size, nkeypoints, input_dim, gaussian_cat_type):
        super().__init__()
        if gaussian_cat_type != "none":
            raise NotImplementedError("gaussian_cat_type other than 'none' is not implemented")
        self.grid_size = grid_size
        self.output_map_width = grid_size // 4
        self.feat_dim = 128
        self.nkeypoints = nkeypoints
        self.gaussian_cat_type = gaussian_cat_type
        self.adjust_combined_representation = nn.Sequential(
            nn.Conv3d(self.feat_dim + 2 * nkeypoints + input_dim, self.feat_dim, kernel_size=1), nn.LeakyReLU())
        self.decode_voxel_from_combined_representation = self.build_voxel_decoder()

    def build_voxel_decoder(self):
        f = self.feat_dim
        up = lambda: nn.Upsample(scale_factor=2.0, mode="trilinear", align_corners=False)  # noqa: E731
        return nn.Sequential(
            up(), nn.Conv3d(f, f // 2, 3, 1, 1), nn.GroupNorm(f // 32, f // 2), nn.LeakyReLU(),
            nn.Conv3d(f // 2, f // 2, 3, 1, 1), nn.GroupNorm(f // 32, f // 2), nn.LeakyReLU(),
            up(), nn.Conv3d(f // 2, f // 4, 3, 1, 1), nn.GroupNorm(f // 64, f // 4), nn.LeakyReLU(),
            nn.Conv3d(f // 4, f // 4, 3, 1, 1), nn.GroupNorm(f // 64, f // 4), nn.LeakyReLU(),
            nn.Conv3d(f // 4, 1, kernel_size=1))

    @staticmethod
    def _conv_after_gn(raw, a, b, conv, gn):
        """conv(LeakyReLU(GroupNorm(raw))): the normalisation is fused into the conv's operand path when the
        kernel supports it, otherwise applied by a separate pass."""
        if ops.can_fuse_input(raw, conv):
            return ops.conv3d(raw, conv, gn, in_affine=(a, b, True))
        return ops.conv3d(ops.affine_act(raw, a, b, True), conv, gn)

    def decode(self, first_feature_act, first_frame, keypoints=None, gaussians=None, sigma=1.5, sharpness=10.0,
               translation=0.5, target=None):
        """first_feature_act (B, g, g, g, 128) act; first_frame (B, 1, G, G, G); keypoints (B, T, K, 4) or
        gaussians (B, T, K, g, g, g); target (B, T, 1, G, G, G) optional -> recon (B, T, 1, G, G, G)
        [, per-frame BCE (B, T)]."""
        _no_training(self)
        src = keypoints if keypoints is not None else gaussians
        B, T = src.shape[:2]
        G, g, K = self.grid_size, self.output_map_width, self.nkeypoints
        dec = self.decode_voxel_from_combined_representation
        dev = first_feature_act.device
        with torch.no_grad():
            first_frame = first_frame.float().contiguous().view(B, G, G, G)
            recon = torch.empty(B, T, 1, G, G, G, dtype=torch.float32, device=dev)
            bce = torch.empty(B, T, dtype=torch.float32, device=dev) if target is not None else None
            if target is not None:
                target = target.float().contiguous()
            clips = max(1, frames_per_pass(G) // T)
            for b0 in range(0, B, clips):
                b1 = min(B, b0 + clips)
                n = (b1 - b0) * T
                kp = keypoints[b0:b1].float().contiguous().view(n, K, 4) if keypoints is not None else None
                gs = gaussians[b0:b1].float().contiguous().view(n, K, g, g, g) if keypoints is None else None
                x = ops.decoder_adjust(first_feature_act[b0:b1], self.adjust_combined_representation[0], T, g, K,
                                       sigma, keypoints=kp, gaussians=gs)
                if UP_DEC1 and ops.can_conv_up2x(x, dec[1]):
                    raw, a, b = ops.conv3d_up2x(x, dec[1], dec[2])     # up-sampling inside the conv's operand path
                else:
                    raw, a, b = ops.conv3d(ops.upsample2x(x), dec[1], dec[2])
                raw, a, b = self._conv_after_gn(raw, a, b, dec[4], dec[5])
                if ops.can_conv_up2x(raw, dec[8]):
                    # GroupNorm + LeakyReLU + trilinear up-sampling all happen inside the conv's operand path: the
                    # 64-channel 64^3 tensor (33.5 MB / frame) is never written
                    raw, a, b = ops.conv3d_up2x(raw, dec[8], dec[9], in_affine=(a, b, True))
                else:
                    x = ops.upsample2x(ops.affine_act(raw, a, b, True))
                    raw, a, b = ops.conv3d(x, dec[8], dec[9])
                raw, a, b = self._conv_after_gn(raw, a, b, dec[11], dec[12])
                tgt = target[b0:b1].view(n, G, G, G) if target is not None else None
                ops.final_recon(raw, a, b, dec[14], first_frame[b0:b1], T, sharpness, translation, target=tgt,
                                out=recon[b0:b1].view(n, G, G, G),
                                bce_out=bce[b0:b1].view(n) if target is not None else None)
            return (recon, bce) if target is not None else recon

    def decode_train(self, first_feature_act, first_frame, keypoints, target, sigma=1.5, sharpness=10.0, translation=0.5):
        """Training-mode `decode` (autograd): keypoints (B, T, K, 4) with graph -> (recon (B, T, 1, G, G, G), BCE (B, T))."""
        B, T = keypoints.shape[:2]
        G, g, K = self.grid_size, self.output_map_width, self.nkeypoints
        dec = self.decode_voxel_from_combined_representation
        adj = self.adjust_combined_representation[0]
        n = B * T
        first_frame = first_frame.detach().float().contiguous().view(B, G, G, G)
        target = target.detach().float().contiguous().view(n, G, G, G)
        x = AG.Adjust.apply(first_feature_act, keypoints.reshape(n, K, 4).contiguous(), adj.weight, adj.bias, adj, T, g, K,
                            sigma)
        x = AG.conv_gn_act(AG.Upsample2x.apply(x), dec[1], dec[2], True)
        x = AG.conv_gn_act(x, dec[4], dec[5], True)
        x = AG.conv_gn_act(AG.Upsample2x.apply(x), dec[8], dec[9], True)
        recon, bce = AG.ConvGNFinalRecon.apply(x, dec[11].weight, dec[11].bias, dec[12].weight, dec[12].bias,
                                               dec[14].weight, dec[14].bias, first_frame, target, dec[11], dec[12],
                                               dec[14], T, sharpness, translation)
        return recon.view(B, T, 1, G, G, G), bce.view(B, T)

    def forward(self, gaussians, first_feature, first_frame, sharpness=10.0, translation=0.5):
        """gaussians (B, T, K, g, g, g), first_feature (B, 128, g, g, g), first_frame (B, 1, G, G, G)."""
        return self.decode(ops.ncdhw_to_act(first_feature), first_frame, gaussians=gaussians, sharpness=sharpness,
                           translation=translation)


class KyptDetector(nn.Module):
    """Detector wrapper: encoder -> decoder -> losses (reference kypt_detector.py:10-241)."""

    def __init__(self, options):
        super().__init__()
        self.vol_fit_type = options.vol_fit_type
        self.fixed_sigma = bool(options.fixed_sigma)
        self.keypoints_graph = options.keypoints_graph
        self.keypoints_detach = bool(options.keypoints_detach)
        self.graph_random_init = bool(options.graph_random_init)
        self.using_local_const = bool(options.using_local_const)
        self.using_time_const = bool(options.using_time_const)
        self.using_sparsity_const = bool(options.using_sparsity_const)
        self.using_intensity_const = bool(options.using_intensity_const)
        self.using_graph_traj = options.graph_traj_weight > 0
        self.using_graph_vol = options.graph_vol_weight > 0
        self.affinity_ver = options.affinity_ver
        self.graph_loss_ver = options.graph_loss_ver
        self.gaussian_sigma = options.gaussian_sigma
        self.is_binarized = options.is_binarized
        self.input_dim = options.input_dim
        self.grid_size = options.grid_size
        self.nkeypoints = options.nkeypoints
        self.sigmas = [self.gaussian_sigma] * self.nkeypoints
        self.vox_to_kypt = VoxToKyptNet(grid_size=options.grid_size, nkeypoints=options.nkeypoints,
                                        input_dim=options.input_dim, sigmas=self.sigmas,
                                        fixed_sigma=bool(options.fixed_sigma),
                                        const_intensity=options.const_intensity)
        self.kypt_to_vox = KyptToVoxNet(grid_size=options.grid_size, nkeypoints=options.nkeypoints,
                                        input_dim=options.input_dim, gaussian_cat_type=options.gaussian_cat_type)
        self.sep_sigma = options.sep_sigma
        self.affinity_anneal = options.affinity_anneal
        self.affinity_start = False
        if self.keypoints_graph == "affinity_params":
            self.nneighbor = options.nneighbor
            cols = self.nkeypoints if self.affinity_ver < 3 else self.nkeypoints - 1
            shape = (self.nneighbor, self.nkeypoints, cols)
            if self.graph_random_init:
                init = torch.randn(*shape)
            else:
                init = torch.zeros(*shape) if self.affinity_ver < 3 else torch.ones(*shape)
            self.affinity_params = nn.Parameter(init)

    def anneal(self, nepoch):
        if self.keypoints_graph != "affinity_params":
            return
        if self.affinity_anneal > nepoch:
            self.affinity_params.requires_grad = False
        elif not self.affinity_start:
            self.affinity_start = True
            self.affinity_params.requires_grad = True

    def get_affinity(self):
        """(nneighbor, K, K, 1) affinity from `affinity_params` (reference kypt_detector.py:171-211)."""
        if self.affinity_ver != 3:
            raise NotImplementedError("only affinity_ver == 3 (the shipped configuration) is implemented")
        K = self.nkeypoints
        w = torch.softmax(self.affinity_params, dim=-1)                      # (n, K, K-1)
        # re-insert a zero diagonal: column j of row i maps to j (j < i) or j + 1 (j >= i)
        upper = torch.cat([torch.zeros_like(w[..., :1]), torch.triu(w, diagonal=0)], dim=-1)
        lower = torch.cat([torch.tril(w, diagonal=-1), torch.zeros_like(w[..., :1])], dim=-1)
        return (upper + lower).unsqueeze(-1)

    def forward_train(self, seq):
        """`forward` with the autograd graph (reference kypt_detector.py:81-169 under `network.train()`): every loss
        term is differentiable w.r.t. the detector parameters it depends on."""
        B, T = seq.shape[:2]
        dev = seq.device
        G, K = self.grid_size, self.nkeypoints
        det = self.vox_to_kypt.detect_train(seq)
        keypoints, heatmaps = det["keypoints"], det["heatmaps"]
        recon, bce = self.kypt_to_vox.decode_train(det["first_feature_act"], seq[:, 0], keypoints, seq,
                                                   sigma=float(self.sigmas[0]))
        zeros = torch.zeros(B, T, device=dev)
        if self.vol_fit_type == "chamfer":
            frames = seq.detach().float().contiguous().view(B * T, G, G, G)
            vol_fit = AG.ChamferVolFit.apply(frames, keypoints.reshape(B * T, K, 4).contiguous()).view(B, T)
        else:
            vol_fit = get_volume_fitting_loss(seq, keypoints, self.vox_to_kypt.sigmas, self.vol_fit_type)
        if self.keypoints_graph == "none" or not self.affinity_start:
            affinity = None
            local = timec = sparse = inten = traj = zeros
        else:
            affinity = self.get_affinity()
            kp_graph = keypoints.detach() if self.keypoints_detach else keypoints
            local, timec, sparse, inten = get_graph_consistency_loss(
                kp_graph, affinity, local_const=self.using_local_const, time_const=self.using_time_const,
                sparsity_const=self.using_sparsity_const, intensity_const=self.using_intensity_const,
                ver=self.graph_loss_ver)
            traj = get_graph_traj_loss(kp_graph, affinity, ver=self.graph_loss_ver) if self.using_graph_traj else zeros
        return dict(
            recon=recon, keypoints=keypoints, heatmaps=heatmaps, affinity=affinity,
            recon_loss=bce.mean(), vol_fit_reg=vol_fit.mean(), kypt_const_loss=zeros.mean(),
            separation_loss=get_temporal_separation_loss(keypoints, self.sep_sigma).mean(),
            sparsity_loss=sparsity_loss_from_means(det["heat_mean"]).mean(),
            local_const_loss=local.mean(), time_const_loss=timec.mean(), sparsity_const_loss=sparse.mean(),
            intensity_const_loss=inten.mean(), graph_traj_loss=traj.mean(), graph_vol_loss=zeros.mean(),
            first_feature=det["first_feature"])

    def forward(self, seq, Tcond=None):
        if not seq.is_cuda:
            raise ops.L.NmError("KyptDetector needs CUDA tensors (there is no CPU fallback)")
        if _training(self):
            return self.forward_train(seq)
        B, T = seq.shape[:2]
        dev = seq.device
        det = self.vox_to_kypt.detect(seq, want_gaussians=False)
        keypoints, heatmaps = det["keypoints"], det["heatmaps"]
        recon, bce = self.kypt_to_vox.decode(det["first_feature_act"], seq[:, 0], keypoints=keypoints,
                                             sigma=float(self.sigmas[0]), target=seq)
        with torch.no_grad():
            zeros = torch.zeros(B, T, device=dev)
            vol_fit = get_volume_fitting_loss(seq, keypoints, self.vox_to_kypt.sigmas, self.vol_fit_type)
            if self.keypoints_graph == "none" or not self.affinity_start:
                affinity = None
                local = timec = sparse = inten = traj = zeros
            else:
                affinity = self.get_affinity()
                local, timec, sparse, inten = get_graph_consistency_loss(
                    keypoints, affinity, local_const=self.using_local_const, time_const=self.using_time_const,
                    sparsity_const=self.using_sparsity_const, intensity_const=self.using_intensity_const,
                    ver=self.graph_loss_ver)
                traj = get_graph_traj_loss(keypoints, affinity, ver=self.graph_loss_ver) if self.using_graph_traj \
                    else zeros
            return dict(
                recon=recon, keypoints=keypoints, heatmaps=heatmaps, affinity=affinity,
                recon_loss=bce.mean(), vol_fit_reg=vol_fit.mean(), kypt_const_loss=zeros.mean(),
                separation_loss=get_temporal_separation_loss(keypoints, self.sep_sigma).mean(),
                sparsity_loss=sparsity_loss_from_means(det["heat_mean"]).mean(),
                local_const_loss=local.mean(), time_const_loss=timec.mean(), sparsity_const_loss=sparse.mean(),
                intensity_const_loss=inten.mean(), graph_traj_loss=traj.mean(), graph_vol_loss=zeros.mean(),
                first_feature=det["first_feature"])

    def decode_from_dyna(self, keypoints, first_feature, first_frame):
        """keypoints (B, Tgen, K, 4), first_feature (B, 128, g, g, g), first_frame (B, 1, G, G, G) -> {'gen'}."""
        gen = self.kypt_to_vox.decode(ops.ncdhw_to_act(first_feature), first_frame, keypoints=keypoints,
                                      sigma=float(self.sigmas[0]))
        return dict(gen=gen)
