"""CPU suite for the host-side logic of the product package and the C-ABI surface (no compute calls)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

from oracle import nm_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from neural_marionette_b200 import _lib
    header = open(os.path.join(ROOT, "include", "nm_b200.h")).read()
    declared = set(re.findall(r"\b(nm_[a-z0-9_]+)\s*\(", header))
    declared.discard("nm_hsvrnn_weights")
    assert declared, "no declarations found"
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for name in sorted(declared):
        assert hasattr(handle, name), f"{name} declared in include/nm_b200.h but not exported"
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert _lib.lib().nm_version() == 100


def test_header_prototypes_match_the_ctypes_bindings():
    """Every declaration of include/nm_b200.h against its ctypes prototype: same number of parameters, and the same kind
    (pointer / int / long long / size_t / float) in every position - an ABI drift between header, library and binding would
    otherwise only show up as garbage arguments on the GPU."""
    from neural_marionette_b200 import _lib
    header = re.sub(r"/\*.*?\*/", " ", open(os.path.join(ROOT, "include", "nm_b200.h")).read(), flags=re.S)
    header = re.sub(r"//[^\n]*", " ", header)
    decls = re.findall(r"\b(?:int|size_t|const char\s*\*)\s+(nm_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", header, flags=re.S)
    assert len(decls) >= 80, len(decls)

    def kind_of_c(param: str) -> str:
        param = " ".join(param.split())
        if "*" in param:
            return "ptr"
        base = param.rsplit(" ", 1)[0] if " " in param else param
        return {"int": "int", "long long": "ll", "size_t": "size", "float": "float", "double": "double",
                "unsigned long long": "ull"}.get(base.replace("const ", ""), base)

    def kind_of_ctypes(t) -> str:
        if isinstance(t, type) and issubclass(t, ctypes._Pointer):
            return "ptr"
        return {ctypes.c_void_p: "ptr", ctypes.c_char_p: "ptr", ctypes.c_int: "int", ctypes.c_longlong: "ll",
                ctypes.c_size_t: "size", ctypes.c_float: "float", ctypes.c_double: "double",
                ctypes.c_ulonglong: "ull"}.get(t, str(t))

    seen = set()
    for name, params in decls:
        plist = [] if params.strip() in ("", "void") else [q for q in params.split(",")]
        assert name in _lib.PROTOTYPES, name
        _, argtypes = _lib.PROTOTYPES[name]
        assert len(plist) == len(argtypes), f"{name}: header has {len(plist)} parameters, the binding {len(argtypes)}"
        for i, (c, t) in enumerate(zip(plist, argtypes)):
            assert kind_of_c(c) == kind_of_ctypes(t), f"{name}: parameter {i} is `{c.strip()}` in the header, {t} in the binding"
        seen.add(name)
    assert seen == set(_lib.PROTOTYPES), seen ^ set(_lib.PROTOTYPES)


def test_state_dict_layout_matches_reference_contract():
    import neural_marionette_b200 as nm
    hp = O.default_hparams()
    net = nm.NeuralMarionette(hp)
    sd = O.synthetic_state_dict(hp, seed=0)       # layout validated against the reference by make_golden.py
    assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v.shape) for k, v in sd.items()}
    assert len(sd) == 337 and sum(v.numel() for v in sd.values()) == 10087015
    assert not net.dyna_module.offset_param.requires_grad
    res = net.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys


def test_affinity_and_skeleton_match_oracle(golden_dir):
    import neural_marionette_b200 as nm
    from neural_marionette_b200.utils.dyna_utils import process_affinity_glob
    hp = O.default_hparams()
    net = nm.NeuralMarionette(hp)
    for c in json.load(open(os.path.join(golden_dir, "skeleton.json"))):
        with torch.no_grad():
            net.kypt_detector.affinity_params.copy_(torch.tensor(c["affinity_params"]))
            aff = net.kypt_detector.get_affinity()
        assert torch.equal(aff, O.get_affinity({"kypt_detector.affinity_params": torch.tensor(c["affinity_params"])}, hp))
        A, pr, pa = process_affinity_glob(aff)
        assert pa.tolist() == c["parents"] and pr.indices.tolist() == c["order"]
        np.testing.assert_allclose(pr.values.numpy(), np.array(c["values"]), rtol=0, atol=1e-12)
        Ao, _, _ = O.skeleton_from_affinity(aff)
        assert torch.equal(A, Ao)


def test_skeleton_random_affinities_match_oracle():
    from neural_marionette_b200.utils.dyna_utils import process_affinity_glob
    hp = O.default_hparams()
    g = torch.Generator().manual_seed(123)
    for trial in range(40):
        sd = {"kypt_detector.affinity_params": torch.randn(2, 24, 23, generator=g) * [0.0, 0.3, 1.0, 4.0][trial % 4]}
        aff = O.get_affinity(sd, hp)
        A, pr, pa = process_affinity_glob(aff)
        Ao, pro, pao = O.skeleton_from_affinity(aff)
        assert torch.equal(pa, pao) and torch.equal(pr.indices, pro.indices) and torch.equal(pr.values, pro.values)
        assert torch.equal(A, Ao)


def test_host_utilities_match_oracle():
    from neural_marionette_b200.utils import dataset_utils as du, geo_utils as gu, kypt_detector_utils as ku
    clip = O.synthetic_clip(7, 3, 500)
    assert np.array_equal(du.episodic_normalization(clip, 0.8, 0.1, 0.0), O.episodic_normalization(clip, 0.8, 0.1, 0.0))
    assert np.array_equal(du.crop_sequence(clip, 1, 2, 1), O.crop_sequence(clip, 1, 2, 1))
    g = torch.Generator().manual_seed(2)
    x = torch.rand(2, 3, 5, 6, 7, generator=g)
    assert torch.equal(ku.add_coord_channels(x), O.add_coord_channels(x))
    hm = torch.nn.functional.softplus(3 * torch.randn(2, 24, 8, 8, 8, generator=g))
    assert (ku.extract_keypoints_from_heatmap(hm) - O.keypoints_from_heatmap(hm)).abs().max() < 1e-6
    p = torch.randn(3, 24, 6, generator=g)
    assert (gu.compute_rotation_matrix_from_6d(p) - O.rot6d_to_matrix(p)).abs().max() < 1e-6
    kp = torch.cat([torch.rand(2, 5, 24, 3, generator=g) - 0.5, torch.rand(2, 5, 24, 1, generator=g)], -1)
    aff = O.get_affinity({"kypt_detector.affinity_params": torch.randn(2, 24, 23, generator=g)}, O.default_hparams())
    a = ku.get_graph_consistency_loss(kp, aff, ver=1)
    b = O.graph_consistency_losses(kp, aff)
    for u, v in zip(a[:3], b[:3]):
        assert (u - v).abs().max() < 1e-6
    assert (ku.get_graph_traj_loss(kp, aff, ver=1) - O.graph_traj_loss(kp, aff)).abs().max() < 1e-6
    assert (ku.get_temporal_separation_loss(kp, 0.02) - O.separation_loss(kp, 0.02)).abs().max() < 1e-6
    hms = torch.rand(2, 5, 24, 4, 4, 4, generator=g)
    assert (ku.get_keypoint_sparsity_loss(hms) - O.sparsity_loss(hms)).abs().max() < 1e-6
    assert (ku.sparsity_loss_from_means(hms.mean(dim=(3, 4, 5))) - O.sparsity_loss(hms)).abs().max() < 1e-6


def test_product_fails_loudly_without_gpu():
    """No CPU fallback: CPU tensors are rejected, a missing library raises."""
    import neural_marionette_b200 as nm
    from neural_marionette_b200 import _lib
    hp = O.default_hparams(grid_size=32)
    net = nm.NeuralMarionette(hp).eval()
    with torch.no_grad(), pytest.raises((_lib.NmError, RuntimeError, AssertionError)):
        net.kypt_detector(torch.zeros(1, 2, 1, 32, 32, 32))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError):
            nm.voxelize(np.zeros((4, 3)), (8, 8, 8))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "neural_marionette_b200")
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(base, f)).read()
                assert "oracle" not in src.replace("the oracle", ""), f"{f} references oracle/"


def test_kernel_choice_ignores_the_environment():
    """Which kernel runs, and what it computes, follows from the arguments alone: no CUDA source reads an environment variable."""
    csrc = os.path.join(ROOT, "neural_marionette_b200", "csrc")
    for base, _, files in os.walk(csrc):
        for f in files:
            if f.endswith((".cu", ".cuh")):
                src = open(os.path.join(base, f)).read()
                assert not re.search(r"\bgetenv\s*\(", src), f"{f} calls getenv"


def test_new_entry_points_reject_cpu_tensors():
    """No CPU fallback anywhere: the §8f#4 consumers and the backward bricks raise on CPU tensors."""
    import numpy as np
    import torch
    from neural_marionette_b200 import _lib, ops
    from collections import namedtuple
    from neural_marionette_b200.utils import retarget_utils as RT
    Priority = namedtuple("Priority", ["values", "indices"])
    a = torch.zeros(1, 8, 8, 8)
    act = torch.zeros(1, 16, 16, 16, 32, dtype=ops.ACT_DTYPE)
    calls = [lambda: ops.voxel_chamfer(a, a.clone()),
             lambda: ops.semantic_nearest(torch.zeros(2, 4, 4), torch.zeros(2, 3, 3)),
             lambda: ops.skin_weights(torch.zeros(5, 3), torch.zeros(4, 4), torch.zeros(4, dtype=torch.int32), 0, 8.0, 0.2),
             lambda: ops.linear_blend_skinning(torch.zeros(5, 3), torch.zeros(4, 3), None, torch.zeros(2, 4, 3, 4), torch.zeros(5, 4)),
             lambda: ops.conv3d_weight_grad(act, act),
             lambda: ops.groupnorm_backward(act, act, torch.nn.GroupNorm(2, 32)),
             lambda: ops.conv3d_input_grad(act, torch.nn.Conv3d(32, 32, 3, 1, 1)),
             lambda: RT.extract_skin_weights(torch.zeros(1), Priority(None, torch.tensor([0, 1])), [0, 0],
                                             np.zeros((3, 3), np.float32), torch.zeros(2, 4))]
    for fn in calls:
        with pytest.raises(_lib.NmError, match="CUDA tensors"):
            fn()
