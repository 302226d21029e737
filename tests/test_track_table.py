"""CPU checks of the device track table (models/tracking.py TrackTable / ReIDTracker): the plain-torch restatement of its
kernels (tests/track_table_reference.py) on hand-made cases of the policy, ReIDTracker with that restatement and the scipy
assignment oracle standing in for the kernels against PointReidentifier.step frame by frame, and the argument handling of the
C entry points (pcreid_track_*), answered before any CUDA call."""
import copy

import pytest
import torch

import assign_blocks_reference as RB
import assign_reference as R
import track_table_reference as TT
from test_multiscene_step import FakeModel, _scene


def _table(S, C, replace_all=False):
    from pcreid_b200.models.tracking import TrackTable
    return TrackTable(S, C, replace_all, device="cpu")


def _dets(labels, lengths=None, boxes=None):
    n = len(labels)
    lengths = [5] * n if lengths is None else lengths
    box = torch.zeros(n, 7) if boxes is None else torch.tensor(boxes, dtype=torch.float32).reshape(n, 7)
    return torch.tensor(labels, dtype=torch.int32), torch.tensor(lengths, dtype=torch.int32), box


def _update(tab, shapes, tfd, dets, max_age=None, replace_all=False):
    return TT.track_update(tab, shapes, torch.tensor(tfd, dtype=torch.int64), *dets, max_age=max_age, replace_all=replace_all)


def _alive_ids(tab, s):
    return tab.tracks(s)[0].tolist()


# ---------------------------------------------------------------------------------------------------------- the policy
def test_slot_freed_and_reused_in_the_same_step():
    tab = _table(1, 2)
    ids, rows = _update(tab, [(0, 2)], [-1, -1], _dets([1, 2]))
    assert ids.tolist() == [0, 1] and rows.tolist() == [0, 1] and tab.count.tolist() == [2]
    # track 0 (slot 0) is left unmatched with max_age 0 and freed; the new detection takes slot 0 in the same step
    ids, rows = _update(tab, [(2, 2)], [1, -1], _dets([2, 3], boxes=[[1.0] * 7, [2.0] * 7]), max_age=0)
    assert ids.tolist() == [1, 2] and rows.tolist() == [1, 0]
    assert tab.track_id[0].tolist() == [2, 1] and tab.label[0].tolist() == [3, 2]
    assert tab.hits[0].tolist() == [1, 2] and tab.age[0].tolist() == [0, 0]
    assert tab.box[0, 1].tolist() == [1.0] * 7 and tab.box[0, 0].tolist() == [2.0] * 7
    assert tab.active[0].tolist() == [0, 1] and tab.next_id.tolist() == [3] and tab.dropped.tolist() == [0]


def test_drops_at_capacity():
    tab = _table(2, 2)
    ids, rows = _update(tab, [(0, 0), (0, 3)], [-1, -1, -1], _dets([0, 0, 0]))
    assert ids.tolist() == [0, 1, -1] and rows.tolist() == [2, 3, -1]
    assert tab.dropped.tolist() == [0, 1] and tab.next_id.tolist() == [0, 2] and tab.count.tolist() == [0, 2]
    # a full scene: every unmatched detection is dropped and next_id does not move
    ids, rows = _update(tab, [(0, 0), (2, 2)], [0, -1], _dets([0, 0]))
    assert ids.tolist() == [0, -1] and rows.tolist() == [2, -1]
    assert tab.dropped.tolist() == [0, 2] and tab.next_id.tolist() == [0, 2]


def test_ids_are_unique_and_never_reused():
    g = torch.Generator().manual_seed(5)
    tab = _table(3, 4)
    seen = [set() for _ in range(3)]
    for _ in range(30):
        shapes, tfd = [], []
        for s in range(3):
            A, D = int(tab.count[s]), int(torch.randint(0, 6, (1,), generator=g))
            pos = torch.randperm(A, generator=g).tolist()[:D]
            col = [pos[d] if d < len(pos) and torch.rand(1, generator=g) < 0.5 else -1 for d in range(D)]
            shapes.append((A, D))
            tfd += col
        n = len(tfd)
        ids, _ = _update(tab, shapes, tfd, _dets([0] * n), max_age=int(torch.randint(0, 3, (1,), generator=g)))
        d0 = 0
        for s, (A, D) in enumerate(shapes):
            for d in range(D):
                i = int(ids[d0 + d])
                if tfd[d0 + d] < 0 and i >= 0:
                    assert i not in seen[s]
                    seen[s].add(i)
            d0 += D
            alive = _alive_ids(tab, s)
            assert len(set(alive)) == len(alive) and all(i in seen[s] for i in alive)
            assert int(tab.next_id[s]) == len(seen[s])
    assert int(tab.dropped.sum()) > 0 and min(len(x) for x in seen) > 4


def test_frozen_scene_and_scene_without_detections():
    tab = _table(2, 4)
    _update(tab, [(0, 2), (0, 2)], [-1] * 4, _dets([0, 1, 0, 1]))
    before = copy.deepcopy(tab)
    # scene 0 has no frame (A = D = 0 though it holds tracks): nothing ages; scene 1 has a frame without detections: all age
    ids, rows = _update(tab, [(0, 0), (2, 0)], [], _dets([]), max_age=5)
    assert ids.numel() == 0 and rows.numel() == 0
    for name in ("alive", "track_id", "age", "hits", "active", "count", "next_id"):
        assert torch.equal(getattr(tab, name)[0], getattr(before, name)[0]), name
    assert tab.age[1, :2].tolist() == [1, 1] and tab.count.tolist() == [2, 2]


def test_max_age_zero_frees_every_unmatched_track():
    tab = _table(1, 3)
    _update(tab, [(0, 3)], [-1, -1, -1], _dets([0, 1, 2]))
    _update(tab, [(3, 1)], [2], _dets([2]), max_age=0)
    assert tab.alive[0].tolist() == [False, False, True] and tab.count.tolist() == [1] and tab.active[0, 0] == 2
    # max_age None: never
    _update(tab, [(1, 0)], [], _dets([]), max_age=None)
    assert tab.alive[0].tolist() == [False, False, True] and tab.age[0, 2] == 1


@pytest.mark.parametrize("replace_all", [False, True])
def test_replace_rule(replace_all):
    tab = _table(1, 2)
    _update(tab, [(0, 2)], [-1, -1], _dets([0, 1], lengths=[10, 10]))
    ids, rows = _update(tab, [(2, 2)], [0, 1], _dets([0, 1], lengths=[3, 10]), replace_all=replace_all)
    assert ids.tolist() == [0, 1]
    # a smaller observation replaces the kept one only with replace_all; an equal one always does
    assert rows.tolist() == ([0, 1] if replace_all else [-1, 1])
    assert tab.length[0].tolist() == ([3, 10] if replace_all else [10, 10])
    assert tab.hits[0].tolist() == [2, 2] and tab.age[0].tolist() == [0, 0]


def test_gate_reference_distance():
    tab = _table(1, 2)
    _update(tab, [(0, 2)], [-1, -1], _dets([1, 1], boxes=[[0.0] * 7, [10.0] * 7]))
    dets = _dets([1, 1, 2], boxes=[[3.0, 4.0] + [0.0] * 5, [3.0, 4.0001] + [0.0] * 5, [0.0] * 7])
    r2 = torch.full((8,), 5.0) ** 2
    g = TT.track_gate_blocks(tab, [(2, 3)], *dets, radius_sq=r2).view(2, 3)
    assert g.tolist() == [[True, False, False], [False, False, False]]       # exactly at the radius passes
    g = TT.track_gate_blocks(tab, [(2, 3)], *dets).view(2, 3)
    assert g.tolist() == [[True, True, False], [True, True, False]]


# ---------------------------------------------------------------------------------------------------------- ReIDTracker
def _patch(monkeypatch):
    import pcreid_b200.kernels as K
    monkeypatch.setattr(K, "linear_assignment", R.linear_assignment)
    monkeypatch.setattr(K, "linear_assignment_blocks", RB.linear_assignment_blocks)
    for name in ("track_gate_blocks", "track_update", "track_scatter"):
        monkeypatch.setattr(K, name, getattr(TT, name))


@pytest.mark.parametrize("replace_all", [False, True])
@pytest.mark.parametrize("min_score", [0.5, -2.0])
def test_tracker_equals_point_reidentifier_step(monkeypatch, replace_all, min_score):
    """S scenes in one ReIDTracker (scene 2 is None in frame 1, scene 3 never has detections) against one PointReidentifier
    per scene called with track_index = arange(len(bank)) and the stored labels: nothing retires, the capacity never fills"""
    import pcreid_b200.models.tracking as TR
    from pcreid_b200.models.tracking import PointFeatureSet, PointReidentifier, ReIDTracker
    _patch(monkeypatch)
    dets = [5, 3, 4, 0]
    S, C = len(dets), 32
    model = FakeModel()
    tracker = ReIDTracker(model, num_scenes=S, capacity=C, replace_all=replace_all, device="cpu")
    banks = [PointFeatureSet(replace_all) for _ in range(S)]
    labels = [torch.zeros(0, dtype=torch.int64) for _ in range(S)]
    matched = 0
    for frame in range(4):
        data = [_scene(s, frame, dets[s], 0) for s in range(S)]
        frames = [None if (s == 2 and frame == 1) else (torch.zeros(0, 4), torch.zeros(dets[s], 7), data[s][2])
                  for s in range(S)]
        live = [s for s in range(S) if frames[s] is not None]
        monkeypatch.setattr(TR, "crop_center_resample_scenes", lambda *a, **kw: (
            torch.cat([data[s][0] for s in live]), torch.cat([data[s][1] for s in live])))
        got = tracker.step(frames, min_score)
        for s in range(S):
            if frames[s] is None:
                assert got[s] is None
                continue
            ref = PointReidentifier(model, banks[s])

            def from_sweep(sweep, bboxes, det_labels, ti, tl, sample_rank=None, ref=ref, s=s):
                xyz_d, h_d = model.encode(data[s][0])
                if ti is None or len(ti) == 0:
                    return None, xyz_d, h_d, data[s][1]
                cost, _, _ = ref(data[s][0], det_labels, data[s][1], ti, tl)
                return cost, xyz_d, h_d, data[s][1]

            monkeypatch.setattr(ref, "from_sweep", from_sweep)
            tfd, new_rows, cost = ref.step(frames[s][0], frames[s][1], data[s][2], torch.arange(len(banks[s])), labels[s],
                                           min_score)
            want = tfd.clone()
            want[tfd < 0] = new_rows
            ids, got_cost = got[s]
            assert torch.equal(ids, want), (frame, s)
            assert (cost is None) == (got_cost is None) and (cost is None or torch.equal(got_cost, cost))
            matched += int((tfd >= 0).sum())
            labels[s] = torch.cat([labels[s], data[s][2][tfd < 0]])
            n = len(banks[s])
            rows = slice(s * C, s * C + n)
            assert tracker.table.count[s] == n and tracker.table.alive[s, :n].all()
            if n:
                assert torch.equal(tracker.table.xyz[rows], banks[s].pts_xyz)
                assert torch.equal(tracker.table.feat[rows], banks[s].pts_feats)
                assert torch.equal(tracker.table.length[s, :n].long(), banks[s].lengths)
                assert torch.equal(tracker.table.label[s, :n].long(), labels[s])
                assert torch.equal(tracker.table.track_id[s, :n], torch.arange(n))
    assert matched > 0


def test_tracker_all_scenes_none_and_bad_arguments():
    from pcreid_b200.models.tracking import ReIDTracker, TrackTable
    tracker = ReIDTracker(FakeModel(), num_scenes=2, capacity=4, device="cpu")
    assert tracker.step([None, None], 0.0) == [None, None]
    with pytest.raises(ValueError):
        tracker.step([None], 0.0)
    for bad in (dict(capacity=0), dict(capacity=4097), dict(max_age=-1), dict(max_distance=[1.0, 2.0]),
                dict(max_distance=-1.0)):
        with pytest.raises(ValueError):
            ReIDTracker(FakeModel(), device="cpu", **bad)
    with pytest.raises(ValueError):
        TrackTable(0, 4, device="cpu")


def test_table_reset_and_tracks():
    tab = _table(2, 3)
    _update(tab, [(0, 2), (0, 1)], [-1, -1, -1], _dets([4, 5, 6], boxes=[[1.0] * 7, [2.0] * 7, [3.0] * 7]))
    ids, labels, boxes, ages, hits, rows = tab.tracks(0)
    assert ids.tolist() == [0, 1] and labels.tolist() == [4, 5] and boxes[:, 0].tolist() == [1.0, 2.0]
    assert ages.tolist() == [0, 0] and hits.tolist() == [1, 1] and rows.tolist() == [0, 1]
    assert tab.tracks(1)[5].tolist() == [3]
    tab.reset(0)
    assert tab.tracks(0)[0].numel() == 0 and tab.next_id.tolist() == [0, 1] and tab.count.tolist() == [0, 1]


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def L():
    from pcreid_b200 import _lib
    return _lib.lib()


def test_track_entry_points_argument_errors_before_any_cuda_call(L):
    gate = lambda S, C, mA, mD, nc=8: L.pcreid_track_gate_blocks(S, C, mA, mD, *([None] * 8), nc, 2, 1, None, None, None)
    for a in ((-1, 4, 1, 1), (1, 0, 1, 1), (1, 4, -1, 1), (1, 4, 1, -1), (1, 4, 5, 1), (1, 4, 1, 1, -1)):
        assert gate(*a) == 1, a
    for a in ((65536, 4, 1, 1), (1, 4097, 1, 1), (1, 4, 1, 4097)):
        assert gate(*a) == 3, a
    assert gate(1, 4, 2, 2) == 1                                     # null pointers
    assert gate(0, 4, 2, 2) == 0 and gate(3, 4, 0, 2) == 0 and gate(3, 4, 2, 0) == 0     # nothing to write
    upd = lambda S, C, mD, max_age=-1: L.pcreid_track_update(S, C, mD, *([None] * 5), max_age, 0, *([None] * 14))
    for a in ((-1, 4, 1), (1, 0, 1), (1, 4, -1), (1, 4, 1, -2)):
        assert upd(*a) == 1, a
    for a in ((65536, 4, 1), (1, 4097, 1), (1, 4, 4097)):
        assert upd(*a) == 3, a
    assert upd(1, 4, 0) == 1 and upd(2, 4, 3, 0) == 1                # null pointers
    assert upd(0, 4, 3) == 0
    sc = L.pcreid_track_scatter
    assert sc(-1, None, 4, None, None, 4, None, None, None) == 1
    assert sc(1, None, -4, None, None, 4, None, None, None) == 1
    assert sc(1, None, 4, None, None, 4, None, None, None) == 1
    assert sc(1, None, 4 << 30, None, None, 4, None, None, None) == 3
    assert sc(0, None, 4, None, None, 4, None, None, None) == 0
    assert sc(3, None, 0, None, None, 0, None, None, None) == 0
