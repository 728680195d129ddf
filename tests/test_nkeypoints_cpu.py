"""Keypoint counts other than 24 on the host: the skeleton built from the affinity, and the constructors' range check."""
import pytest
import torch

from oracle import nm_oracle as O


@pytest.mark.parametrize("K", [16, 45, 64])
def test_skeleton_random_affinities_match_oracle(K):
    from neural_marionette_b200.utils.dyna_utils import process_affinity_glob
    hp = O.default_hparams(nkeypoints=K)
    g = torch.Generator().manual_seed(K)
    for trial in range(12):
        sd = {"kypt_detector.affinity_params": torch.randn(2, K, K - 1, generator=g) * [0.0, 0.3, 1.0, 4.0][trial % 4]}
        aff = O.get_affinity(sd, hp)
        A, pr, pa = process_affinity_glob(aff)
        Ao, pro, pao = O.skeleton_from_affinity(aff)
        assert torch.equal(pa, pao) and torch.equal(pr.indices, pro.indices) and torch.equal(pr.values, pro.values)
        assert torch.equal(A, Ao)


@pytest.mark.parametrize("K", [1, 65, 96])
def test_constructors_reject_out_of_range_nkeypoints(K):
    from neural_marionette_b200.model.hsvrnn_bvh import HSVRNNBVH
    from neural_marionette_b200.model.kypt_detector import KyptDetector
    hp = O.default_hparams(nkeypoints=K)
    with pytest.raises(NotImplementedError, match="nkeypoints"):
        KyptDetector(hp)
    with pytest.raises(NotImplementedError, match="nkeypoints"):
        HSVRNNBVH(hp)


@pytest.mark.parametrize("K", [2, 24, 64])
def test_constructors_accept_the_supported_range(K):
    from neural_marionette_b200.model.hsvrnn_bvh import HSVRNNBVH
    from neural_marionette_b200.model.kypt_detector import KyptDetector
    hp = O.default_hparams(nkeypoints=K)
    assert KyptDetector(hp).nkeypoints == K
    assert HSVRNNBVH(hp).root_intensity_decoder[2].out_features == 3 + K
