"""CPU checks of the bank bookkeeping of PointReidentifier.step (models/tracking.py): the sweep -> cost part (from_sweep) is
replaced by fixed tensors and kernels.linear_assignment by the scipy oracle (tests/assign_reference.py)."""
import copy

import numpy as np
import pytest
import torch

import assign_reference


def _bank(replace_all, n=5, seed=0):
    from pcreid_b200.models.tracking import PointFeatureSet
    g = torch.Generator().manual_seed(seed)
    bank = PointFeatureSet(replace_all)
    bank.store_new(torch.randn(n, 16, 3, generator=g), torch.randn(n, 8, 16, generator=g), torch.tensor([10, 50, 30, 40, 60])[:n])
    return bank


def _reid(monkeypatch, bank, frame):
    """a PointReidentifier whose from_sweep returns `frame` = (cost, xyz_d, h_d, len_d)."""
    import pcreid_b200.kernels as K
    from pcreid_b200.models.tracking import PointReidentifier
    monkeypatch.setattr(K, "linear_assignment", assign_reference.linear_assignment)
    reid = PointReidentifier(None, bank)
    monkeypatch.setattr(reid, "from_sweep", lambda *args, **kw: frame)
    return reid


def _detections(D, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(D, 16, 3, generator=g), torch.randn(D, 8, 16, generator=g)


@pytest.mark.parametrize("replace_all", [False, True])
@pytest.mark.parametrize("min_score", [0.2, -0.5])
def test_step_matched_replace_unmatched_store(monkeypatch, replace_all, min_score):
    bank = _bank(replace_all)
    before = copy.deepcopy(bank)
    track_index = torch.tensor([4, 1, 2])
    track_labels = torch.tensor([0, 1, 0])
    det_labels = torch.tensor([0, 1, 2, 0])
    det_len = torch.tensor([20, 40, 60, 5])
    # zeros where the class gate forbids the pair: with min_score < 0 they would be worth matching without the gate
    cost = torch.tensor([[2.0, 0.0, 0.0, 0.5],
                         [0.0, 1.0, 0.0, 0.0],
                         [1.5, 0.0, 0.0, 1.8]])
    xyz_d, h_d = _detections(4)
    reid = _reid(monkeypatch, bank, (cost, xyz_d, h_d, det_len))
    track_for_det, new_rows, got_cost = reid.step(None, None, det_labels, track_index, track_labels, min_score)
    assert track_for_det.dtype == torch.long and track_for_det.tolist() == [0, 1, -1, 2]
    assert new_rows.dtype == torch.long and new_rows.tolist() == [5]
    assert got_cost is cost
    # det 0 -> bank row 4 (60 points) holds 60 >= 20: kept unless replace_all; det 1 -> row 1 (50 > 40): the same;
    # det 3 -> row 2 (30 > 5): the same.  A replaced row holds the detection's tensors.
    replaced = {4: 0, 1: 1, 2: 3} if replace_all else {}
    for row in range(5):
        src = (xyz_d[replaced[row]], h_d[replaced[row]], det_len[replaced[row]]) if row in replaced else \
            (before.pts_xyz[row], before.pts_feats[row], before.lengths[row])
        assert torch.equal(bank.pts_xyz[row], src[0]) and torch.equal(bank.pts_feats[row], src[1])
        assert torch.equal(bank.lengths[row], src[2])
    assert len(bank) == 6
    assert torch.equal(bank.pts_xyz[5], xyz_d[2]) and torch.equal(bank.pts_feats[5], h_d[2]) and int(bank.lengths[5]) == 60


def test_step_replaces_when_the_new_observation_has_more_points(monkeypatch):
    bank = _bank(False)
    cost = torch.tensor([[1.0, 3.0]])
    xyz_d, h_d = _detections(2)
    reid = _reid(monkeypatch, bank, (cost, xyz_d, h_d, torch.tensor([100, 10])))
    track_for_det, new_rows, _ = reid.step(None, None, torch.tensor([0, 0]), torch.tensor([0]), torch.tensor([0]), 0.0)
    assert track_for_det.tolist() == [-1, 0] and new_rows.tolist() == [5]
    assert int(bank.lengths[0]) == 10 and torch.equal(bank.pts_feats[0], h_d[1])       # 10 >= 10 points: replaced
    assert int(bank.lengths[5]) == 100 and torch.equal(bank.pts_xyz[5], xyz_d[0])


def test_step_without_active_tracks_stores_every_detection(monkeypatch):
    bank = _bank(False, n=3)
    xyz_d, h_d = _detections(4)
    det_len = torch.tensor([3, 4, 5, 6])
    reid = _reid(monkeypatch, bank, (None, xyz_d, h_d, det_len))
    track_for_det, new_rows, cost = reid.step(None, None, torch.zeros(4, dtype=torch.long), torch.zeros(0, dtype=torch.long),
                                              torch.zeros(0, dtype=torch.long), 0.0)
    assert cost is None and track_for_det.tolist() == [-1] * 4 and new_rows.tolist() == [3, 4, 5, 6]
    assert torch.equal(bank.pts_feats[3:], h_d) and torch.equal(bank.pts_xyz[3:], xyz_d) and torch.equal(bank.lengths[3:], det_len)
    # and into an empty bank
    from pcreid_b200.models.tracking import PointFeatureSet
    empty = PointFeatureSet()
    reid = _reid(monkeypatch, empty, (None, xyz_d, h_d, det_len))
    _, new_rows, _ = reid.step(None, None, torch.zeros(4, dtype=torch.long), None, None, 0.0)
    assert new_rows.tolist() == [0, 1, 2, 3] and torch.equal(empty.pts_feats, h_d)


@pytest.mark.parametrize("replace_all", [False, True])
def test_step_equals_manual_composition_on_random_frames(monkeypatch, replace_all):
    from pcreid_b200.models.tracking import class_gate
    rng = np.random.default_rng(3)
    bank = _bank(replace_all)
    manual = copy.deepcopy(bank)
    for frame in range(3):
        T, D = len(bank), int(rng.integers(1, 8))
        track_index = torch.from_numpy(rng.permutation(T)[:max(1, T - 2)])
        tl = torch.from_numpy(rng.integers(0, 3, track_index.numel()))
        dl = torch.from_numpy(rng.integers(0, 3, D))
        det_len = torch.from_numpy(rng.integers(0, 80, D))
        gate = class_gate(dl, tl, det_len, manual.lengths[track_index])
        cost = torch.where(gate, torch.from_numpy(rng.normal(size=gate.shape).astype(np.float32)), torch.zeros(()))
        xyz_d, h_d = _detections(D, seed=10 + frame)
        reid = _reid(monkeypatch, bank, (cost, xyz_d, h_d, det_len))
        track_for_det, new_rows, _ = reid.step(None, None, dl, track_index, tl, -0.25)
        # by hand: oracle + the bank's own methods
        _, t4d = assign_reference.assign(cost.numpy(), np.float32(-0.25), gate.numpy())
        assert track_for_det.tolist() == t4d.tolist()
        m, u = np.nonzero(t4d >= 0)[0], np.nonzero(t4d < 0)[0]
        manual.replace_old(track_index[t4d[m]], xyz_d[m], h_d[m], det_len[m])
        first = len(manual)
        manual.store_new(xyz_d[u], h_d[u], det_len[u])
        assert new_rows.tolist() == list(range(first, first + len(u)))
        assert torch.equal(bank.pts_xyz, manual.pts_xyz) and torch.equal(bank.pts_feats, manual.pts_feats)
        assert torch.equal(bank.lengths, manual.lengths)
