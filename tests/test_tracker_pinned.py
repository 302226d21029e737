"""Pins the all-pairs driver pieces (SURVEY 8f row 1) to the reference's OWN deprecated tracker files, imported unmodified by
path (oracle/ref_loader.load_tracker): get_labels_to_compare (tracking_point_reid.py:15-33) against the oracle's / product's
dense class gate, PointFeatureSet (tracking_feature_set.py:12-63) against the product's feature bank."""
import pytest
import torch

from oracle import ref_loader, reid_oracle as O

pytestmark = pytest.mark.skipif(not ref_loader.tracker_available(), reason=ref_loader.MISSING)


@pytest.fixture(scope="module")
def R():
    return ref_loader.load_tracker()


@pytest.mark.parametrize("seed,use_lengths", [(0, True), (1, True), (2, False), (3, True)])
def test_class_gate_vs_reference_get_labels_to_compare(R, seed, use_lengths):
    from pcreid_b200.models.tracking import class_gate
    g = torch.Generator().manual_seed(seed)
    T, D = 23, 17
    tl, dl = torch.randint(0, 11, (T,), generator=g), torch.randint(0, 11, (D,), generator=g)      # classes 8..10 are never compared
    tn, dn = torch.randint(0, 6, (T,), generator=g), torch.randint(0, 6, (D,), generator=g)        # < 2 points: never compared
    if seed == 3:
        tl[:] = 9                                                                                   # nothing to compare -> None
    pairs = R.get_labels_to_compare(dl, tl, dn, tn, use_lengths, 'cpu')
    ref = torch.zeros(T, D, dtype=torch.bool)
    if pairs is not None:
        ref[pairs[:, 0], pairs[:, 1]] = True
        assert pairs.shape[0] == int(ref.sum())                 # no duplicates in the reference list
    else:
        assert seed == 3
    assert torch.equal(ref, class_gate(dl, tl, dn, tn, use_lengths=use_lengths))
    if use_lengths:
        assert torch.equal(ref, O.class_gated_pairs(tl, tn, dl, dn))


@pytest.mark.parametrize("replace_all", [False, True])
def test_feature_bank_vs_reference_point_feature_set(R, replace_all):
    from pcreid_b200.models.tracking import PointFeatureSet
    g = torch.Generator().manual_seed(7)
    ref, mine = R.PointFeatureSet(replace_all), PointFeatureSet(replace_all)
    with pytest.raises(ValueError):
        ref.replace_old(torch.tensor([0]), None, None, None)
    with pytest.raises(ValueError):
        mine.replace_old(torch.tensor([0]), None, None, None)
    for step in range(6):
        n = 3 + step
        xyz, feats = torch.randn(n, 16, 3, generator=g), torch.randn(n, 8, 16, generator=g)
        lengths = torch.randint(0, 50, (n,), generator=g)
        if step % 2 == 0:
            ref.store_new(xyz.clone(), feats.clone(), lengths.clone())
            mine.store_new(xyz.clone(), feats.clone(), lengths.clone())
        else:
            index = torch.randperm(ref.pts_feats.shape[0], generator=g)[:n]
            m = index.numel()
            ref.replace_old(index, xyz[:m].clone(), feats[:m].clone(), lengths[:m].clone())
            mine.replace_old(index, xyz[:m].clone(), feats[:m].clone(), lengths[:m].clone())
        assert torch.equal(ref.pts_feats, mine.pts_feats) and torch.equal(ref.pts_xyz, mine.pts_xyz)
        assert torch.equal(ref.lengths, mine.lengths)
    idx = torch.tensor([4, 0, 2])
    assert all(torch.equal(a, b) for a, b in zip(ref.get_features(idx), mine.get_features(idx)))
    ref.reset()
    mine.reset()
    assert ref.pts_feats is None and mine.pts_feats is None
