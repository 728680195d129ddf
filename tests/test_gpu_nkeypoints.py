"""Keypoint counts other than the shipped 24 (nkeypoints in 2..64) on the GPU, against the CPU oracle at the tolerances
of the K = 24 tests.  K <= 24 runs the tuned kernel instantiations, 24 < K <= 64 a second set compiled for 64; the K
values cover both sides, multiples and non-multiples of 8 and of 4, and the maximum."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import nm_oracle as O

import test_gpu_dyna_train as DT
from test_gpu_kernels import from_act, rel_err, to_act
from test_gpu_model import HM_TOL, KP_TOL, clips

pytestmark = pytest.mark.gpu

KS = [16, 21, 32, 45, 64]
Z = 128


@pytest.fixture(scope="module")
def ops():
    from neural_marionette_b200 import ops as _ops
    return _ops


def _net(K, seed, G=32, train=False):
    import neural_marionette_b200 as nm
    hp = O.default_hparams(grid_size=G, nkeypoints=K)
    sd = O.synthetic_state_dict(hp, seed=seed)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().train(train)
    net.anneal(1)
    return net, sd, hp


def _kp(gen, B, T, K, spread=1.2):
    return torch.cat([torch.rand(B, T, K, 3, generator=gen) * spread - spread / 2, torch.rand(B, T, K, 1, generator=gen)], -1)


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("K", KS)
def test_heatmap_head_softargmax_render(ops, K):
    g = 16
    gen = torch.Generator().manual_seed(K)
    C, B, T = 128, 2, 3
    conv1 = torch.nn.Conv3d(C, K, 1)
    prop = torch.nn.Conv3d(2, 1, 1)
    with torch.no_grad():
        conv1.weight.mul_(6.0)
        prop.weight.copy_(torch.tensor([1.5, 0.75]).view(1, 2, 1, 1, 1))
        prop.bias.fill_(-1.0)
    feat = torch.randn(B * T, C, g, g, g, generator=gen)
    prev = torch.randn(B, K, g, g, g, generator=gen)
    hm = F.leaky_relu(conv1(feat.half().float()), 0.01).reshape(B * T * K, 1, g, g, g)
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
    conv2 = torch.nn.Conv3d(256, K, 1)
    f2 = torch.randn(2, 256, g, g, g, generator=gen)
    ref = F.leaky_relu(conv2(f2.half().float()), 0.01).detach()
    assert rel_err(ops.heatmap_head(to_act(f2), conv2.cuda(), K, 0).cpu(), ref) < 1e-4
    assert (ops.gaussian_render(kp.cuda(), 1.5, g).cpu() - gs).abs().max() < 2e-4


@pytest.mark.parametrize("K", KS)
def test_decoder_adjust(ops, K):
    gen = torch.Generator().manual_seed(100 + K)
    B, T, g = 2, 3, 8
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


@pytest.mark.parametrize("K", KS)
def test_chamfer(ops, K):
    gen = torch.Generator().manual_seed(200 + K)
    seq = (torch.rand(2, 3, 1, 16, 16, 16, generator=gen) < 0.05).float()
    kp = torch.cat([torch.rand(2, 3, K, 3, generator=gen) * 2 - 1, torch.rand(2, 3, K, 1, generator=gen)], -1)
    ref = O.chamfer_vol_fit(seq, kp)
    got = ops.chamfer_vol_fit(seq.reshape(6, 16, 16, 16).cuda(), kp.reshape(6, K, 4).cuda()).view(2, 3).cpu()
    assert (got - ref).abs().max() < 1e-5


# ------------------------------------------------------------------------------------------------ detector
@pytest.mark.parametrize("K,G", [(k, 32) for k in KS] + [(64, 64)])
def test_detector_vs_oracle(K, G):
    B, T = 2, 3
    net, sd, hp = _net(K, 300 + K, G)
    vox, vox_ref = clips(6000 + K, B, T, 20000, G)
    with torch.no_grad():
        out = net.kypt_detector(vox)
        ref = O.detector_forward(vox_ref, sd, hp)
        gen_kp = out["keypoints"][:, :1].contiguous()
        gen = net.kypt_detector.decode_from_dyna(gen_kp, out["first_feature"], vox[:, 0])["gen"]
    assert out["keypoints"].shape == (B, T, K, 4)
    assert (out["keypoints"].cpu() - ref["keypoints"]).abs().max() <= KP_TOL
    assert float((out["heatmaps"].cpu() - ref["heatmaps"]).abs().max() / ref["heatmaps"].max()) <= HM_TOL
    assert (out["recon"].cpu() - ref["recon"]).abs().mean() <= 5e-3
    assert (gen.cpu() - ref["recon"][:, :1]).abs().mean() <= 5e-3


# ------------------------------------------------------------------------------------------------ dynamics
@pytest.mark.parametrize("K", KS)
def test_dynamics_encode_generate_vs_oracle(K):
    net, sd, hp = _net(K, 400 + K)
    gen = torch.Generator().manual_seed(K)
    B, T = 3, 5
    kp = _kp(gen, B, T, K)
    eps = torch.randn(T, 10, B, Z, generator=gen)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        skel = O.skeleton_from_affinity(aff.cpu())
        got = net.dyna_module.encode(kp.cuda(), aff, eps=eps.cuda())
        ref = O.dyna_encode(kp, skel, sd, hp, eps=eps)
    for k in ["kypt_recon", "R", "z_kypts", "h_kypts"]:
        assert (got[k].cpu() - ref[k]).abs().max() < 5e-4, k
    assert abs(float(got["kl_kypt"]) - float(ref["kl_kypt"])) < 1e-3 * abs(float(ref["kl_kypt"]))
    # generate: the conditioned steps equal encode's, the free-running ones are deterministic given the draws
    ec = torch.randn(2, 10, B, Z, generator=gen)
    eg = torch.randn(3, B, Z, generator=gen)
    with torch.no_grad():
        out = net.dyna_module.generate(kp[:, :2].cuda(), aff, Ttot=5, Tcond=2, eps_cond=ec.cuda(), eps_gen=eg.cuda())
        ref2 = O.dyna_encode(kp[:, :2], skel, sd, hp, eps=ec)
        again = net.dyna_module.generate(kp[:, :2].cuda(), aff, Ttot=5, Tcond=2, eps_cond=ec.cuda(), eps_gen=eg.cuda())
    assert out["keypoints_gen"].shape == (B, 3, K, 4)
    assert (out["keypoints_cond"].cpu() - ref2["kypt_recon"]).abs().max() < 5e-4
    assert torch.isfinite(out["keypoints_gen"]).all()
    assert torch.equal(out["keypoints_gen"], again["keypoints_gen"])


@pytest.mark.parametrize("K", KS)
def test_dynamics_interpolate_vs_oracle(K):
    net, sd, hp = _net(K, 500 + K)
    gen = torch.Generator().manual_seed(50 + K)
    T, sample_num, sample_rate = 7, 6, 3
    kp = _kp(gen, 1, T, K)
    eps = torch.randn(T, 2, sample_num, Z, generator=gen)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        out = net.dyna_module.interpolate(kp.cuda(), aff, sample_num=sample_num, sample_rate=sample_rate, eps=eps.cuda())
        sel, picks = O.dyna_interpolate(kp, O.skeleton_from_affinity(aff.cpu()), sd, hp, sample_num, sample_rate, eps)
    assert out["picks"].cpu().tolist() == torch.as_tensor(picks).tolist()
    assert (out["keypoints"].cpu() - sel).abs().max() < 5e-4


@pytest.mark.parametrize("K", [21, 64])
def test_dynamics_large_batch_matches_small(K):
    """At K = 21 the small batch runs the cluster kernel; at K = 64 every batch runs the one-CTA-per-element kernel
    (the cluster layout does not fit).  The large batch runs one CTA per element or per four elements."""
    net, sd, hp = _net(K, 600 + K)
    gen = torch.Generator().manual_seed(K)
    B = 640
    kp = _kp(gen, B, 2, K, 1.0).cuda()
    ec = torch.randn(2, 10, B, Z, generator=gen).cuda()
    eg = torch.randn(2, B, Z, generator=gen).cuda()
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
        net.dyna_module.encode(kp[:2], aff)             # builds the skeleton
        big = net.dyna_module.generate(kp, aff, Ttot=4, Tcond=2, eps_cond=ec, eps_gen=eg)
        small = net.dyna_module.generate(kp[:40], aff, Ttot=4, Tcond=2, eps_cond=ec[:, :, :40].contiguous(),
                                         eps_gen=eg[:, :40].contiguous())
    assert (big["keypoints_gen"][:40] - small["keypoints_gen"]).abs().max() < 1e-4
    assert (big["keypoints_cond"][:40] - small["keypoints_cond"]).abs().max() < 1e-4


# ------------------------------------------------------------------------------------------------ stage 2
@pytest.mark.parametrize("K", [16, 45, 64])
def test_encode_gradients_match_float64_autograd(K):
    B, T, seed = 5, 6, 700 + K
    net, sd, hp = _net(K, seed, train=True)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
    gen = torch.Generator().manual_seed(seed)
    kp, eps = _kp(gen, B, T, K), torch.randn(T, 10, B, Z, generator=gen)
    names = DT._dyna_names(False)
    out, got = DT._run_gpu(net, kp, eps, aff, DT._probe(DT._shapes(B, T, K), seed))
    ref, want, sd64 = DT._oracle_grads(kp, eps, aff, sd, hp, DT._probe(DT._shapes(B, T, K), seed), names)
    assert (out["z_kypts"].detach().cpu().double() - ref["z_kypts"]).abs().max() < 5e-4, "picks differ from the oracle"
    gaps = DT._pick_gaps(ref, kp, eps, aff, sd64)
    assert float(gaps.min()) > 1e-5, f"near-tie between the two best samples: relative gap {float(gaps.min()):.2e}"
    report, whole = DT._compare(got, want, names)
    bad = {n: v for n, v in report.items() if v[0] > 1e-3 or v[1] < 0.9999}
    assert not bad, bad
    assert whole <= 1e-4, (whole, report)
    # bit-reproducible
    _, again = DT._run_gpu(net, kp, eps, aff, DT._probe(DT._shapes(B, T, K), seed))
    for n in names:
        assert torch.equal(got[n], again[n]), n


@pytest.mark.parametrize("K", [32, 64])
def test_stage2_adam_loop_decreases_loss(K):
    from neural_marionette_b200.optim import FusedAdam
    net, sd, hp = _net(K, 800 + K, train=True)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
    gen = torch.Generator().manual_seed(K)
    B, T = 24, 20
    kp = _kp(gen, B, T, K, 1.0).cuda()
    dm = net.dyna_module
    opt = FusedAdam([p for p in dm.parameters() if p.requires_grad], lr=1e-3)
    losses = []
    for _ in range(15):
        opt.zero_grad(set_to_none=True)
        out = dm.encode(kp, aff)
        loss = out["kypt_recon_loss"] + 1e-3 * out["kl_kypt"]
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert all(np.isfinite(losses))
    assert losses[-1] < losses[0], losses


# ------------------------------------------------------------------------------------------------ rejection
def test_k65_is_rejected():
    import neural_marionette_b200 as nm
    from neural_marionette_b200 import _lib, ops
    hp = O.default_hparams(grid_size=32, nkeypoints=65)
    with pytest.raises(NotImplementedError, match="nkeypoints"):
        nm.NeuralMarionette(hp)
    kp = torch.zeros(1, 65, 4, device="cuda")
    with pytest.raises(_lib.NmError, match="K=65"):
        ops.gaussian_render(kp, 1.5, 8)


# ------------------------------------------------------------------------------------------------ backward kernels
from oracle import nm_oracle_eval as E                          # noqa: E402
from oracle import nm_oracle_grad as OG                         # noqa: E402
from test_gpu_backward import WHOLE_TOL, _head_setup, h         # noqa: E402


@pytest.mark.parametrize("K", KS)
def test_heatmap_head_backward(ops, K):
    import copy
    from neural_marionette_b200 import autograd as AG
    B, T, g = 2, 3, 8
    gen, feat, fst, head, hst, prop = _head_setup(21 + K, B, T, g, K)
    n = B * T
    dkp = torch.randn(n, K, 4, generator=gen)
    dhm = torch.randn(n, K, generator=gen)
    feat_r, fst_r = feat.clone().requires_grad_(True), fst.clone().requires_grad_(True)
    prev = F.leaky_relu(hst(fst_r), 0.01)
    u = F.leaky_relu(head(feat_r), 0.01).view(n * K, 1, g, g, g)
    pv = prev.repeat_interleave(T, 0).reshape(n * K, 1, g, g, g)
    hm = F.softplus(prop(torch.cat([u, pv], 1))).view(n, K, g, g, g)
    kp = O.keypoints_from_heatmap(hm)
    ((kp * dkp).sum() + (hm.mean(dim=(2, 3, 4)) * dhm).sum()).backward()
    ref_grads = {k: v.grad.clone() for k, v in dict(hw=head.weight, hb=head.bias, sw=hst.weight, sb=hst.bias,
                                                    pw=prop.weight, pb=prop.bias).items()}
    head_c, hst_c, prop_c = (copy.deepcopy(m).cuda() for m in (head, hst, prop))
    for p in list(head_c.parameters()) + list(hst_c.parameters()) + list(prop_c.parameters()):
        p.grad = None
    ops.set_grad_scale(256.0)
    fa = to_act(feat).requires_grad_(True)
    fs = to_act(fst).requires_grad_(True)
    link = {}
    prev_c = AG.HeadST.apply(fs, hst_c.weight, hst_c.bias, hst_c, K, link)
    heat_c, kp_c, mean_c = AG.Head.apply(fa, head_c.weight, head_c.bias, prev_c, prop_c.weight, prop_c.bias, head_c, prop_c,
                                         K, T, 1.5, link)
    assert float((kp_c.detach().cpu() - kp.detach()).abs().max()) < 1e-4
    ((kp_c * dkp.cuda()).sum() + (mean_c * dhm.cuda()).sum()).backward()
    assert rel_err(from_act(fa.grad) / 256.0, feat_r.grad) < 3e-3
    assert rel_err(from_act(fs.grad) / 256.0, fst_r.grad) < 3e-3
    got = dict(hw=head_c.weight.grad, hb=head_c.bias.grad, sw=hst_c.weight.grad, sb=hst_c.bias.grad, pw=prop_c.weight.grad,
               pb=prop_c.bias.grad)
    for k in ref_grads:
        assert rel_err(got[k].cpu(), ref_grads[k]) < 2e-3, k


@pytest.mark.parametrize("K", KS)
def test_decoder_adjust_backward(ops, K):
    import copy
    from neural_marionette_b200 import autograd as AG
    gen = torch.Generator().manual_seed(33 + K)
    B, T, g = 2, 3, 8
    n = B * T
    ff = h(torch.randn(B, 128, g, g, g, generator=gen))
    kp = torch.cat([torch.rand(n, K, 3, generator=gen) * 1.4 - 0.7, torch.rand(n, K, 1, generator=gen) * 0.8 + 0.2], -1)
    conv = torch.nn.Conv3d(128 + 2 * K + 3, 128, 1)
    with torch.no_grad():
        conv.weight.copy_(torch.randn(conv.weight.shape, generator=gen) / (128 + 2 * K + 3) ** 0.5)
    gy = h(torch.randn(n, 128, g, g, g, generator=gen))
    ff_r, kp_r = ff.clone().requires_grad_(True), kp.clone().requires_grad_(True)
    gs = O.render_gaussians(kp_r, 1.5, g).view(B, T, K, g, g, g)
    outs = [conv(O.add_coord_channels(torch.cat([gs[:, t], ff_r, gs[:, 0]], 1))) for t in range(T)]
    conv_c = copy.deepcopy(conv).cuda()
    ops.set_grad_scale(64.0)
    ffa = to_act(ff).requires_grad_(True)
    kpc = kp.cuda().requires_grad_(True)
    yc = AG.Adjust.apply(ffa, kpc, conv_c.weight, conv_c.bias, conv_c, T, g, K, 1.5)
    mask = torch.where(from_act(yc.detach()) > 0, 1.0, 0.01)
    y = torch.stack(outs, 1).reshape(n, 128, g, g, g) * mask
    (y * gy).sum().backward()
    assert rel_err(from_act(yc), y.detach()) < 5e-3
    yc.backward((to_act(gy).float() * 64.0).half())
    assert rel_err(from_act(ffa.grad) / 64.0, ff_r.grad) < 3e-3
    assert rel_err(kpc.grad.cpu(), kp_r.grad) < 3e-3
    assert rel_err(conv_c.weight.grad.cpu(), conv.weight.grad) < 3e-3
    assert rel_err(conv_c.bias.grad.cpu(), conv.bias.grad) < 3e-3


@pytest.mark.parametrize("K", KS)
def test_chamfer_backward(ops, K):
    gen = torch.Generator().manual_seed(44 + K)
    B, T, G = 2, 2, 16
    seq = (torch.rand(B, T, 1, G, G, G, generator=gen) < 0.08).float()
    kp = torch.cat([torch.rand(B, T, K, 3, generator=gen) * 1.6 - 0.8, torch.rand(B, T, K, 1, generator=gen)], -1)
    kp_r = kp.clone().requires_grad_(True)
    go = torch.rand(B, T, generator=gen) + 0.5
    (O.chamfer_vol_fit(seq, kp_r) * go).sum().backward()
    got = ops.chamfer_vol_fit_backward(seq.view(B * T, G, G, G).cuda(), kp.view(B * T, K, 4).cuda(), go.view(-1).cuda())
    assert rel_err(got.cpu().view(B, T, K, 4), kp_r.grad) < 1e-4


# ------------------------------------------------------------------------------------------------ stage 1
@pytest.mark.parametrize("K", KS)
def test_training_step_gradients(K):
    """Every trainable detector tensor gets a finite gradient; the reconstruction-loss gradient agrees with the fp32
    oracle on the whole-gradient level (as test_training_step_other_shapes at K = 24)."""
    import neural_marionette_b200 as nm
    G, B, T = 32, 2, 3
    hp = O.default_hparams(grid_size=G, Tcond=3, Ttot=10, nkeypoints=K)
    sd = O.synthetic_state_dict(hp, seed=90 + K)
    vox = torch.from_numpy(np.stack([O.voxelize_clip(O.episodic_normalization(O.synthetic_clip(950 + b, T, 5000)), G)
                                     for b in range(B)], 0)).float()
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().train()
    net.anneal(1)
    out = net.kypt_detector(vox.cuda())
    OG.detector_loss(out, recon_only=True).backward()
    grads = {"kypt_detector." + k: p.grad.detach().float().cpu() for k, p in net.kypt_detector.named_parameters()
             if p.grad is not None}
    assert len(grads) == 314 and all(torch.isfinite(g).all() for g in grads.values())
    _, ref = OG.detector_gradients(vox, sd, hp, recon_only=True)
    allg = torch.cat([grads[k].double().reshape(-1) for k in sorted(grads)])
    allr = torch.cat([ref[k].double().reshape(-1) for k in sorted(grads)])
    err = float((allg - allr).norm() / allr.norm())
    print(f"[K={K}] whole-gradient relative L2 error {err:.3e}")
    assert err <= WHOLE_TOL


# ------------------------------------------------------------------------------------------------ graphs
def test_captured_detector_from_points_k64():
    from neural_marionette_b200 import graph as NG
    import neural_marionette_b200 as nm
    G, T, K = 32, 4, 64
    net, _, _ = _net(K, 53, G)
    det = net.kypt_detector
    raw_a = torch.from_numpy(O.synthetic_clip(8100, T, 20000))[None].cuda()
    raw_b = torch.from_numpy(O.synthetic_clip(8101, T, 20000))[None].cuda()
    with torch.no_grad():
        eager_b = det(nm.voxelize_raw_clips(raw_b, G))
    cap = NG.capture_detector_from_points(det, raw_a, G)
    for _ in range(2):
        got = cap(raw_b)
        for key in ("keypoints", "heatmaps", "recon", "recon_loss", "vol_fit_reg"):
            assert torch.equal(got[key], eager_b[key]), key


def test_captured_train_step_k64():
    """Two replays of `graph.CapturedTrainStep` equal two eager steps with `FusedAdam.step_device()` bit for bit."""
    import neural_marionette_b200 as nm
    from neural_marionette_b200 import graph, ops, optim
    G, B, T, N, K = 32, 2, 3, 4000, 64
    hp = O.default_hparams(grid_size=G, Tcond=3, Ttot=10, nkeypoints=K)
    sd = O.synthetic_state_dict(hp, seed=5)
    raw = torch.from_numpy(np.stack([O.synthetic_clip(300 + b, T, N) for b in range(B)], 0)).cuda()
    loss_fn = lambda out: OG.detector_loss(out, recon_only=False)    # noqa: E731

    def fresh():
        net = nm.NeuralMarionette(hp)
        net.load_state_dict(sd, strict=True)
        net = net.cuda().train()
        net.anneal(1)
        return net, optim.FusedAdam(net.kypt_detector.parameters(), lr=4e-4, owner=net)

    results = {}
    for mode in ("device", "graph"):
        net, opt = fresh()
        losses = []
        if mode == "graph":
            step = graph.CapturedTrainStep(net.kypt_detector, opt, loss_fn, raw, G, warmup=2)
            for _ in range(2):
                losses.append(float(step(raw)))
        else:
            for _ in range(4):
                vox = ops.normalize_voxelize(raw, G, check=False)
                opt.zero_grad()
                loss = loss_fn(net.kypt_detector(vox))
                loss.backward()
                opt.step_device()
                losses.append(float(loss.detach()))
        results[mode] = (losses, torch.cat([p.detach().reshape(-1) for p in net.kypt_detector.parameters()]).clone())
    assert results["graph"][0][-2:] == results["device"][0][2:]
    assert torch.equal(results["graph"][1], results["device"][1])


# ------------------------------------------------------------------------------------------------ retargeting
def test_retargeting_on_a_k64_skeleton():
    """Skin weights, FK and LBS on the skeleton of a K = 64 model against the oracle's restatements."""
    from collections import namedtuple
    from neural_marionette_b200.utils import retarget_utils as RT
    Priority = namedtuple("Priority", ["values", "indices"])
    K = 64
    net, sd, hp = _net(K, 61)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
    _, pr, parents = O.skeleton_from_affinity(aff.cpu())
    order = pr.indices
    gen = torch.Generator().manual_seed(61)
    kp = _kp(gen, 1, 1, K, 1.2)[0, 0]
    pts = (torch.rand(3000, 3, generator=gen) * 1.4 - 0.7).numpy()
    w = RT.extract_skin_weights(torch.zeros(1).cuda(), Priority(None, order), parents, pts, kp.cuda(), 8.0, 0.2)
    ref = E.extract_skin_weights(order, parents, pts, kp)
    same_bone = ((w != 0) == (ref != 0)).all(1)
    assert same_bone.mean() >= 0.999
    assert np.abs(w[same_bone] - ref[same_bone]).max() <= 2e-6
    Tn = 3
    R = torch.linalg.qr(torch.randn(Tn, K, 3, 3, generator=gen))[0]
    off = torch.randn(K, 3, generator=gen) * 0.1
    root = torch.randn(Tn, 3, generator=gen) * 0.1
    src = torch.zeros(1, Tn, K, 4)
    src[0, :, int(order[0]), :3] = root
    src[..., 3] = 0.7
    new_kp = RT.retarget_keypoints(R.cuda(), off.cuda().view(1, -1, 3, 1), src.cuda(), Priority(None, order), parents)
    want = E.retarget_fk(R, off, root, order, parents)
    assert np.abs(new_kp[0, ..., :3].cpu().numpy() - want.numpy()).max() <= 1e-5
    pos = want
    T3x4 = np.concatenate([R.numpy(), pos.numpy()[..., None]], -1)
    lbs_ref = E.linear_blend_skinning(pts, kp[:, :3].numpy(), None, T3x4, ref)
    out = RT.linear_blend_skinning(pts, kp[:, :3].numpy(), None, R.cuda(), pos.cuda(), ref)
    assert np.abs(out - lbs_ref).max() <= 2e-5
