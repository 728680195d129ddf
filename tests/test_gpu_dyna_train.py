"""Stage 2 of the reference's training (train.py:146-147): gradients of `HSVRNNBVH.encode` on the CUDA backward
(`nm_hsvrnn_step_backward` per step, `nm_hsvrnn_weight_grads` once), checked against autograd over the CPU restatement
run in float64."""
import numpy as np
import pytest
import torch

from oracle import nm_oracle as O

PREFIX = "dyna_module"
Z = 128


def _setup(seed, train=True):
    import neural_marionette_b200 as nm
    hp = O.default_hparams()
    sd = O.synthetic_state_dict(hp, seed=seed)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().train(train)
    net.anneal(1)
    with torch.no_grad():
        aff = net.kypt_detector.get_affinity()
    return net, sd, hp, aff


def _inputs(seed, B, T, K=24, S=10):
    gen = torch.Generator().manual_seed(seed)
    kp = torch.cat([torch.rand(B, T, K, 3, generator=gen) * 1.2 - 0.6, torch.rand(B, T, K, 1, generator=gen)], -1)
    eps = torch.randn(T, S, B, Z, generator=gen)
    return kp, eps


OUT_KEYS = ["kypt_recon", "R", "z_kypts", "h_kypts", "kl_kypt", "kypt_recon_loss"]


def _probe(out, seed):
    """Fixed random directions for the weighted sum of all six differentiable outputs."""
    gen = torch.Generator().manual_seed(seed)
    return {k: (torch.randn(tuple(out[k].shape), generator=gen, dtype=torch.float64), 0.5 + i * 0.25)
            for i, k in enumerate(OUT_KEYS)}


def _loss(out, probe):
    total = 0.0
    for k, (g, w) in probe.items():
        total = total + w * (out[k] * g.to(device=out[k].device, dtype=out[k].dtype)).sum()
    return total


def _dyna_names(with_offset):
    names = []
    for mod in ["extract_post_dist", "extract_prior_dist", "root_intensity_decoder", "joint_matrix_decoder"]:
        for layer in (0, 2):
            names += [f"{mod}.{layer}.weight", f"{mod}.{layer}.bias"]
    names += ["kypt_rnn_cell.weight_ih", "kypt_rnn_cell.weight_hh", "kypt_rnn_cell.bias_ih", "kypt_rnn_cell.bias_hh",
              "init_kypt_rnn_state"]
    return names + (["offset_param"] if with_offset else [])


def _oracle_grads(kp, eps, aff, sd, hp, probe, names):
    """float64 autograd over O.dyna_encode (decode_pose builds `pos` with the default dtype: set it to float64)."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        sd64 = {k: v.detach().double() for k, v in sd.items()}
        leaves = [sd64[PREFIX + "." + n].requires_grad_(True) for n in names]
        ref = O.dyna_encode(kp.double(), O.skeleton_from_affinity(aff.cpu()), sd64, hp, eps=eps.double())
        grads = torch.autograd.grad(_loss(ref, probe), leaves)
    finally:
        torch.set_default_dtype(old)
    return ref, dict(zip(names, grads)), sd64


def _pick_gaps(ref, kp, eps, aff, sd64):
    """Relative gap between the best and the second-best sample distance of every (b, t), on the float64 restatement."""
    _, priority, parents = O.skeleton_from_affinity(aff.cpu())
    B, T, K, _ = kp.shape
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        with torch.no_grad():
            kp = kp.double()
            offset = O.bone_offsets(kp, parents, sd64, PREFIX)
            gaps = torch.empty(B, T, dtype=torch.float64)
            for t in range(T):
                h = ref["h_kypts"][:, t]
                kpf = kp[:, t].reshape(B, -1)
                post = O._mlp(torch.cat([h, kpf], -1), sd64, PREFIX + ".extract_post_dist")
                mean, std = post[:, :Z], torch.nn.functional.softplus(post[:, Z:]) + 1e-4
                d = torch.stack([(kpf - O.decode_pose(torch.cat([h, mean + std * eps[t, s].double()], -1), offset,
                                                     priority.indices, parents, sd64, K, PREFIX)[0]).pow(2).sum(-1)
                                 for s in range(eps.shape[1])], 0)
                top = d.sort(dim=0).values
                gaps[:, t] = (top[1] - top[0]) / top[0]
    finally:
        torch.set_default_dtype(old)
    return gaps


def _compare(got, ref, names):
    num = den = 0.0
    report = {}
    for n in names:
        g, r = got[n].double().cpu().reshape(-1), ref[n].reshape(-1)
        rel = float((g - r).norm() / r.norm().clamp_min(1e-30))
        cos = float(torch.dot(g, r) / (g.norm() * r.norm()).clamp_min(1e-30))
        report[n] = (rel, cos)
        num += float((g - r).pow(2).sum())
        den += float(r.pow(2).sum())
    return report, (num / den) ** 0.5


def _run_gpu(net, kp, eps, aff, probe, with_offset=False):
    dm = net.dyna_module
    for p in dm.parameters():
        p.grad = None
    out = dm.encode(kp.cuda(), aff, eps=eps.cuda())
    _loss(out, probe).backward()
    params = dict(dm.named_parameters())
    return out, {n: params[n].grad for n in _dyna_names(with_offset)}


# B = 1 / 5 / 24 / 96 run the cluster kernel forward, B = 100 the one-CTA-per-element kernel, B = 600 the four-elements-per-CTA
# kernel on 148 SMs; the backward splits columns over CTAs and elements over 16-row tiles (1, 2 and 38 tiles here)
@pytest.mark.gpu
@pytest.mark.parametrize("B,T,seed", [(1, 5, 41), (5, 7, 42), (24, 20, 43), (100, 3, 44), (600, 2, 45)])
def test_encode_gradients_match_float64_autograd(B, T, seed):
    net, sd, hp, aff = _setup(seed)
    kp, eps = _inputs(seed + 100, B, T)
    names = _dyna_names(False)
    out, got = _run_gpu(net, kp, eps, aff, _probe(_shapes(B, T), seed))
    ref, want, sd64 = _oracle_grads(kp, eps, aff, sd, hp, _probe(_shapes(B, T), seed), names)
    assert (out["z_kypts"].detach().cpu().double() - ref["z_kypts"]).abs().max() < 5e-4, "picks differ from the oracle"
    gaps = _pick_gaps(ref, kp, eps, aff, sd64)
    assert float(gaps.min()) > 1e-5, f"near-tie between the two best samples: relative gap {float(gaps.min()):.2e}"
    report, whole = _compare(got, want, names)
    bad = {n: v for n, v in report.items() if v[0] > 1e-3 or v[1] < 0.9999}
    assert not bad, bad
    assert whole <= 1e-4, (whole, report)
    assert net.dyna_module.offset_param.grad is None


def _shapes(B, T, K=24):
    return {"kypt_recon": torch.zeros(B, T, K, 4), "R": torch.zeros(B, T, K, 3, 3), "z_kypts": torch.zeros(B, T, Z),
            "h_kypts": torch.zeros(B, T + 1, 512), "kl_kypt": torch.zeros(()), "kypt_recon_loss": torch.zeros(())}


@pytest.mark.gpu
def test_offset_param_gradient_after_learner_reactivation():
    net, sd, hp, aff = _setup(46)
    kp, eps = _inputs(146, 5, 6)
    probe = _probe(_shapes(5, 6), 46)
    _run_gpu(net, kp, eps, aff, probe)
    assert net.dyna_module.offset_param.grad is None                  # the reference's default: frozen
    net.control_active({"detector": True, "learner": False})
    net.control_active({"detector": True, "learner": True})
    assert net.dyna_module.offset_param.requires_grad
    names = _dyna_names(True)
    _, got = _run_gpu(net, kp, eps, aff, probe, with_offset=True)
    _, want, _ = _oracle_grads(kp, eps, aff, sd, hp, probe, names)
    report, whole = _compare(got, want, names)
    bad = {n: v for n, v in report.items() if v[0] > 1e-3 or v[1] < 0.9999}
    assert not bad, bad
    assert whole <= 1e-4, (whole, report)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [3, 100])
def test_training_forward_is_the_eval_forward(B):
    net, sd, hp, aff = _setup(47)
    kp, eps = _inputs(147, B, 4)
    dm = net.dyna_module
    with torch.no_grad():
        ref = dm.encode(kp.cuda(), aff, eps=eps.cuda())
    got = dm.encode(kp.cuda(), aff, eps=eps.cuda())
    assert got["h_kypts"].requires_grad
    for k in OUT_KEYS:
        assert torch.equal(got[k].detach(), ref[k]), k
    torch.manual_seed(3)
    a = dm.encode(kp.cuda(), aff)
    torch.manual_seed(3)
    with torch.no_grad():
        b = dm.encode(kp.cuda(), aff)
    assert torch.equal(a["z_kypts"].detach(), b["z_kypts"])


@pytest.mark.gpu
def test_backward_is_bit_reproducible():
    net, sd, hp, aff = _setup(48)
    kp, eps = _inputs(148, 24, 8)
    probe = _probe(_shapes(24, 8), 48)
    _, g1 = _run_gpu(net, kp, eps, aff, probe)
    g1 = {n: g.clone() for n, g in g1.items()}
    _, g2 = _run_gpu(net, kp, eps, aff, probe)
    for n in g1:
        assert torch.equal(g1[n], g2[n]), n


@pytest.mark.gpu
def test_forward_and_backward_never_synchronise():
    net, sd, hp, aff = _setup(49)
    kp, eps = _inputs(149, 24, 20)
    kp, eps = kp.cuda(), eps.cuda()
    dm = net.dyna_module
    out = dm.encode(kp, aff, eps=eps)              # builds the skeleton and the weight caches
    (out["kypt_recon_loss"] + out["kl_kypt"]).backward()
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = dm.encode(kp, aff, eps=eps)
        (out["kypt_recon_loss"] + out["kl_kypt"]).backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()


def _clips(B, T, G):
    import neural_marionette_b200 as nm
    raw = np.stack([O.synthetic_clip(700 + b, T, 8000) for b in range(B)], 0)
    return nm.voxelize_raw_clips(raw, G)


def _stage2_run(kind, vox, steps=30):
    import neural_marionette_b200 as nm
    from neural_marionette_b200 import optim
    hp = O.default_hparams(grid_size=32)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(O.synthetic_state_dict(hp, seed=50), strict=True)
    net = net.cuda().train()
    net.anneal(1)
    act = {"detector": False, "learner": True}
    net.control_active(act)
    params = net.dyna_module.parameters()
    opt = optim.FusedAdam(params, lr=4e-4, owner=net) if kind == "fused" else \
        torch.optim.Adam([p for p in params if p.requires_grad], lr=4e-4)
    losses = []
    torch.manual_seed(0)
    for _ in range(steps):
        opt.zero_grad()
        out = net(vox, act)
        loss = out["kypt_recon_loss"] + out["kl_kypt"]
        loss.backward()
        opt.step()
        losses.append(float(loss))
    return losses, [p.detach().clone() for p in net.dyna_module.parameters()]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["fused", "torch"])
def test_stage2_training_loop(kind):
    vox = _clips(2, 6, 32)
    l1, p1 = _stage2_run(kind, vox)
    l2, p2 = _stage2_run(kind, vox)
    assert l1[-1] < l1[0], l1
    assert l1 == l2
    assert all(torch.equal(a, b) for a, b in zip(p1, p2))


@pytest.mark.gpu
def test_joint_step_reaches_every_trainable_parameter():
    import neural_marionette_b200 as nm
    from oracle import nm_oracle_grad as OG
    hp = O.default_hparams(grid_size=32)
    net = nm.NeuralMarionette(hp)
    net.load_state_dict(O.synthetic_state_dict(hp, seed=51), strict=True)
    net = net.cuda().train()
    net.anneal(1)
    act = {"detector": True, "learner": True}
    out = net(_clips(2, 6, 32), act)
    (OG.detector_loss(out, recon_only=False) + out["kypt_recon_loss"] + out["kl_kypt"]).backward()
    missing = [n for n, p in net.named_parameters() if p.requires_grad and (p.grad is None or not torch.isfinite(p.grad).all())]
    assert not missing, missing
    assert net.dyna_module.init_kypt_rnn_state.grad.abs().sum() > 0


@pytest.mark.gpu
def test_guards():
    net, sd, hp, aff = _setup(52)
    kp, eps = _inputs(152, 2, 3)
    dm = net.dyna_module
    with pytest.raises(NotImplementedError):
        dm.encode(kp.cuda().requires_grad_(True), aff, eps=eps.cuda())
    dm.encode(kp.cuda(), aff, eps=eps.cuda())
    with pytest.raises(NotImplementedError):
        dm.generate(kp.cuda(), aff, Ttot=5, Tcond=2)
    with pytest.raises(NotImplementedError):
        dm.interpolate(kp[:1].cuda(), aff)


def test_stage2_entry_points_reject_cpu_tensors():
    from neural_marionette_b200 import _lib, ops
    t = torch.zeros(2, 4)
    i = torch.zeros(2, dtype=torch.int32)
    with pytest.raises(_lib.NmError, match="CUDA tensors"):
        ops.hsvrnn_step_record(None, t, t, t, t, i, i, 1, t, t, t, t, t, t, i)
    with pytest.raises(_lib.NmError, match="CUDA tensors"):
        ops.hsvrnn_step_backward(None, None, t, t, t, i, t, t, t, t, i, i, 1, t, t, t, t, t, t, t, t, t, t)
    with pytest.raises(_lib.NmError, match="CUDA tensors"):
        ops.hsvrnn_weight_grads(t, t, t, t, t, t, t, t, None, [t] * 22)
