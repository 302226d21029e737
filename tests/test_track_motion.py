"""CPU checks of the track table's motion (models/tracking.py MotionModel, kernels.track_predict / track_correct /
track_gate_motion_blocks): the 13-value covariance of tests/track_motion_reference.py against the textbook 10 x 10 Kalman
filter in float64, the yaw rules by hand, the bookkeeping around freed, dropped and frozen slots, ReIDTracker(motion=...) with
the CPU restatements standing in for the kernels, and the argument handling of the C entry points."""
import math
import types

import numpy as np
import pytest
import torch

import assign_blocks_reference as RB
import track_motion_reference as TM
import track_table_reference as TT
from test_multiscene_step import FakeModel, _scene

F32 = lambda v: float(np.float32(v))          # noqa: E731  (a parameter as the kernels receive it)


def _table(S, C):
    from pcreid_b200.models.tracking import TrackTable
    return TrackTable(S, C, device="cpu", motion=True)


def _dets(boxes):
    box = torch.tensor(boxes, dtype=torch.float32).reshape(-1, 7)
    n = box.shape[0]
    return torch.zeros(n, dtype=torch.int32), torch.full((n,), 5, dtype=torch.int32), box


# ---------------------------------------------------------------------------------------------------------- exactness
class FullKalman:
    """the textbook filter on the 10-vector (x, y, z, dx, dy, dz, yaw, vx, vy, vz): F, Q, H, R, P0 as matrices (AB3DMOT)"""

    def __init__(self, z, init_var, init_vel_var, q, q_vel, r):
        self.x = np.concatenate([z, np.zeros(3)])
        self.P = np.diag([init_var] * 7 + [init_vel_var] * 3)
        self.Q = np.diag([q] * 7 + [q_vel] * 3)
        self.H = np.hstack([np.eye(7), np.zeros((7, 3))])
        self.R = r * np.eye(7)

    def predict(self, dt):
        F = np.eye(10)
        F[0, 7] = F[1, 8] = F[2, 9] = dt
        self.x = F @ self.x
        self.P = F @ self.P @ F.T + self.Q

    def correct(self, z):
        y = z - self.H @ self.x
        y[6] = (y[6] + math.pi) % (2 * math.pi) - math.pi               # AB3DMOT's orientation correction
        if abs(y[6]) > math.pi / 2:
            y[6] = (y[6] + 2 * math.pi) % (2 * math.pi) - math.pi
        S = self.H @ self.P @ self.H.T + self.R
        K = self.P @ self.H.T @ np.linalg.inv(S)
        self.x = self.x + K @ y
        self.P = (np.eye(10) - K @ self.H) @ self.P

    def compact(self):
        P = self.P
        return np.array([v for a in range(3) for v in (P[a, a], P[a, 7 + a], P[7 + a, 7 + a])] + [P[k, k] for k in range(3, 7)])


def _close(got, want):
    scale = max(1.0, float(np.abs(want).max()))
    assert float(np.abs(got - want).max()) <= 1e-9 * scale, (got, want)


def test_compact_covariance_equals_the_full_filter():
    rng = np.random.default_rng(0)
    C = 4
    par = dict(init_var=F32(10), init_vel_var=F32(1e4), q=F32(1), q_vel=F32(0.01), r=F32(1))
    f64 = torch.float64
    tab = types.SimpleNamespace(active=torch.arange(C, dtype=torch.int32)[None], kf_box=torch.zeros(1, C, 7, dtype=f64),
                                kf_vel=torch.zeros(1, C, 3, dtype=f64), kf_cov=torch.zeros(1, C, 13, dtype=f64))
    truth = rng.uniform(-20, 20, (C, 7))
    truth[:, 6] = rng.uniform(-0.3, 0.3, C)
    vel = rng.uniform(-3, 3, (C, 3))
    z0 = truth + rng.normal(0, 0.3, (C, 7))
    TM.track_correct(tab, [(0, C)], torch.zeros(0, dtype=torch.long), torch.full((C,), -1), torch.from_numpy(z0).float(),
                     torch.arange(C, dtype=torch.int32), par["init_var"], par["init_vel_var"], par["r"])
    full = [FullKalman(z0[i].astype(np.float32).astype(np.float64), **par) for i in range(C)]
    corrections = 0
    for step in range(50):
        dt = F32(0.0 if step % 13 == 5 else rng.uniform(0.05, 2.0))
        TM.track_predict(tab, [(C, 0)], dt, par["q"], par["q_vel"])
        for f in full:
            f.predict(dt)
        truth[:, :3] += dt * vel
        seen = [i for i in range(C) if rng.random() < 0.7]               # the others miss this step
        z = (truth[seen] + rng.normal(0, 0.3, (len(seen), 7))).astype(np.float32)
        z[:, 6] = rng.uniform(-0.3, 0.3, len(seen))
        TM.track_correct(tab, [(C, len(seen))], torch.arange(C), torch.tensor(seen, dtype=torch.long),
                         torch.from_numpy(z), torch.full((len(seen),), -1, dtype=torch.int32), par["init_var"],
                         par["init_vel_var"], par["r"])
        for k, i in enumerate(seen):
            full[i].correct(z[k].astype(np.float64))
        corrections += len(seen)
        for i, f in enumerate(full):
            _close(tab.kf_box[0, i].numpy(), f.x[:7])
            _close(tab.kf_vel[0, i].numpy(), f.x[7:])
            _close(tab.kf_cov[0, i].numpy(), f.compact())
            # nothing else of the 10 x 10 covariance is ever coupled
            kept = np.zeros((10, 10), bool)
            for a in range(3):
                kept[a, a] = kept[a, 7 + a] = kept[7 + a, a] = kept[7 + a, 7 + a] = True
            for k in range(3, 7):
                kept[k, k] = True
            assert float(np.abs(f.P[~kept]).max()) <= 1e-12 * float(np.abs(f.P).max())
    assert corrections > 100


# ---------------------------------------------------------------------------------------------------------- yaw by hand
def _wrap64(a):
    return a - 2 * math.pi * round(a / (2 * math.pi))


def test_yaw_rules_by_hand():
    # (estimate, detection yaw, estimate after the correction with gain 1/2)
    half = math.pi / 2
    cases = [(0.0, half + 0.01, 0.5 * (half + 0.01 - math.pi)),          # just above pi/2: the heading is flipped
             (0.0, half - 0.01, 0.5 * (half - 0.01)),                    # just below: as it is
             (0.0, -half - 0.01, 0.5 * (-half - 0.01 + math.pi)),
             (0.0, -half + 0.01, 0.5 * (-half + 0.01)),
             (3.0, -2.9, _wrap64(3.0 + 0.5 * _wrap64(-5.9))),             # across +-pi, both ways
             (-3.0, 2.9, _wrap64(-3.0 + 0.5 * _wrap64(5.9))),
             (0.2, 2 * math.pi + 0.3, 0.25),                             # a detection yaw outside (-pi, pi]
             (0.2, -4 * math.pi + 0.3, 0.25)]
    n = len(cases)
    tab = _table(1, n)
    tab.active[0] = torch.arange(n, dtype=torch.int32)
    tab.kf_cov.fill_(1.0)                                                # P = r = 1: gain 1/2
    tab.kf_box[0, :, 6] = torch.tensor([c[0] for c in cases])
    z = torch.zeros(n, 7)
    z[:, 6] = torch.tensor([c[1] for c in cases])
    TM.track_correct(tab, [(n, n)], torch.arange(n), torch.arange(n), z, torch.full((n,), -1, dtype=torch.int32), r=1.0)
    got = tab.kf_box[0, :, 6].tolist()
    for (est, det, want), g in zip(cases, got):
        assert abs(g - want) < 2e-6, (est, det, g, want)
        assert -math.pi <= g <= math.pi
    assert got[4] < -3.0 and got[5] > 3.0                                 # the estimate crossed +-pi
    assert tab.kf_cov[0, :, 12].tolist() == [0.5] * n
    # births: the detection's yaw, wrapped
    yaws = [4.0, -7.0, 0.5, 2 * math.pi + 0.3, -math.pi + 1e-3]
    tab = _table(1, len(yaws))
    zb = torch.zeros(len(yaws), 7)
    zb[:, 6] = torch.tensor(yaws)
    TM.track_correct(tab, [(0, len(yaws))], torch.zeros(0, dtype=torch.long), torch.full((len(yaws),), -1), zb,
                     torch.arange(len(yaws), dtype=torch.int32))
    for y, g in zip(yaws, tab.kf_box[0, :, 6].tolist()):
        assert abs(g - _wrap64(y)) < 2e-6 and -math.pi < g <= math.pi, (y, g)


# ---------------------------------------------------------------------------------------------------------- bookkeeping
P0 = [10.0, 0.0, 1e4] * 3 + [10.0] * 4


def test_slot_freed_and_reborn_gets_fresh_motion_state():
    tab = _table(1, 2)
    dets = _dets([[0.0] * 7, [5.0] * 6 + [0.1]])
    _, rows = TT.track_update(tab, [(0, 2)], torch.tensor([-1, -1]), *dets)
    TM.track_correct(tab, [(0, 2)], torch.zeros(0, dtype=torch.long), torch.tensor([-1, -1]), dets[2], rows)
    assert tab.kf_cov[0, 0].tolist() == P0 and tab.kf_box[0, 1].tolist() == dets[2][1].tolist()
    tab.kf_vel[0] = 2.0
    TM.track_predict(tab, [(2, 2)], 1.0)
    track_rows = tab.active[0, :2].long().clone()
    # slot 0 goes unmatched with max_age 0 and is freed; detection 1 is born into it in the same step
    dets = _dets([[6.0] * 6 + [0.2], [9.0] * 6 + [4.0]])
    tfd = torch.tensor([1, -1])
    _, rows = TT.track_update(tab, [(2, 2)], tfd, *dets, max_age=0)
    assert rows.tolist() == [1, 0]
    TM.track_correct(tab, [(2, 2)], track_rows, tfd, dets[2], rows)
    assert tab.kf_box[0, 0, :6].tolist() == [9.0] * 6 and abs(float(tab.kf_box[0, 0, 6]) - _wrap64(4.0)) < 1e-6
    assert tab.kf_vel[0, 0].tolist() == [0.0] * 3 and tab.kf_cov[0, 0].tolist() == P0
    assert tab.kf_vel[0, 1].tolist() != [2.0] * 3 and tab.kf_cov[0, 1, 0] < 10.0      # slot 1 was corrected


def test_dropped_detections_and_unmatched_tracks_touch_nothing():
    tab = _table(1, 2)
    dets = _dets([[1.0] * 7, [2.0] * 7])
    _, rows = TT.track_update(tab, [(0, 2)], torch.tensor([-1, -1]), *dets)
    TM.track_correct(tab, [(0, 2)], torch.zeros(0, dtype=torch.long), torch.tensor([-1, -1]), dets[2], rows)
    TM.track_predict(tab, [(2, 2)], 0.5)
    before = [t.clone() for t in (tab.kf_box, tab.kf_vel, tab.kf_cov)]
    track_rows = tab.active[0, :2].long().clone()
    # the scene is full: detection 1 is dropped; track 1 goes unmatched
    dets = _dets([[1.5] * 7, [30.0] * 7])
    tfd = torch.tensor([0, -1])
    ids, rows = TT.track_update(tab, [(2, 2)], tfd, *dets)
    assert ids.tolist() == [0, -1] and rows.tolist() == [0, -1] and tab.dropped.tolist() == [1]
    TM.track_correct(tab, [(2, 2)], track_rows, tfd, dets[2], rows)
    for t, b in zip((tab.kf_box, tab.kf_vel, tab.kf_cov), before):
        assert torch.equal(t[0, 1], b[0, 1]) and not torch.equal(t[0, 0], b[0, 0])


def test_frozen_scene_is_not_predicted_and_dt_zero_adds_only_noise():
    tab = _table(2, 3)
    dets = _dets([[1.0] * 7, [2.0] * 7, [3.0] * 7, [4.0] * 7])
    _, rows = TT.track_update(tab, [(0, 2), (0, 2)], torch.full((4,), -1), *dets)
    TM.track_correct(tab, [(0, 2), (0, 2)], torch.zeros(0, dtype=torch.long), torch.full((4,), -1), dets[2], rows)
    tab.kf_vel.fill_(1.5)
    tab.kf_cov[..., 1] = 0.25
    before = [t.clone() for t in (tab.kf_box, tab.kf_vel, tab.kf_cov)]
    TM.track_predict(tab, [(0, 0), (2, 1)], [7.0, 0.0], q=0.5, q_vel=0.125)
    for t, b in zip((tab.kf_box, tab.kf_vel, tab.kf_cov), before):
        assert torch.equal(t[0], b[0])                                   # scene 0 has no frame: its dt is not used
    assert torch.equal(tab.kf_box[1], before[0][1]) and torch.equal(tab.kf_vel[1], before[1][1])
    want = before[2][1, :2].clone()
    want[:, [0, 3, 6]] += 0.5
    want[:, [2, 5, 8]] += 0.125
    want[:, 9:] += 0.5
    assert torch.equal(tab.kf_cov[1, :2], want)
    TM.track_predict(tab, [(0, 0), (2, 1)], [0.0, 2.0])
    assert torch.equal(tab.kf_box[1, :2, :3], before[0][1, :2, :3] + 3.0)


def test_gate_reference_uses_the_predicted_box_and_the_mahalanobis_bound():
    tab = _table(1, 1)
    dets = _dets([[0.0] * 7])
    _, rows = TT.track_update(tab, [(0, 1)], torch.tensor([-1]), *dets)
    TM.track_correct(tab, [(0, 1)], torch.zeros(0, dtype=torch.long), torch.tensor([-1]), dets[2], rows)
    tab.kf_vel[0, 0] = torch.tensor([3.0, 4.0, 0.0])
    TM.track_predict(tab, [(1, 0)], 1.0, q=0.0, q_vel=0.0)
    assert tab.kf_box[0, 0, :2].tolist() == [3.0, 4.0]
    tab.kf_cov[0, 0, 0], tab.kf_cov[0, 0, 3] = 2.0, 4.0                 # Sx = 3, Sy = 5 with r = 1
    q = _dets([[3.0, 4.0] + [0.0] * 5, [0.0] * 7, [6.0, 4.0] + [0.0] * 5, [6.0, 9.0] + [0.0] * 5])
    r2 = torch.full((8,), 25.0)
    g = TM.track_gate_motion_blocks(tab, [(1, 4)], *q, radius_sq=r2).tolist()
    assert g == [True, True, True, False]                               # radius 5 around (3, 4), exactly at it passes
    # d^2 = 0, 9/3 + 16/5, 9/3 and 9/3 + 25/5 = 8
    for chi2, want in ((8.0, [True] * 4), (7.999, [True, True, True, False]), (5.0, [True, False, True, False])):
        assert TM.track_gate_motion_blocks(tab, [(1, 4)], *q, r=1.0, gate_chi2=chi2).tolist() == want, chi2
    assert TM.track_gate_motion_blocks(tab, [(1, 4)], *q, radius_sq=r2, gate_chi2=5.0).tolist() == [True, False, True, False]


# ---------------------------------------------------------------------------------------------------------- ReIDTracker
def _patch(monkeypatch, calls):
    import pcreid_b200.kernels as K

    def log(name, fn):
        def wrapped(*a, **kw):
            calls.append(name)
            return fn(*a, **kw)
        return wrapped
    monkeypatch.setattr(K, "linear_assignment_blocks", log("assign", RB.linear_assignment_blocks))
    for mod, names in ((TT, ("track_gate_blocks", "track_update", "track_scatter")),
                       (TM, ("track_predict", "track_correct", "track_gate_motion_blocks"))):
        for name in names:
            monkeypatch.setattr(K, name, log(name, getattr(mod, name)))


def _run(monkeypatch, tracker, dets, frames_n, dt=lambda frame: 1.0):
    import pcreid_b200.models.tracking as TR
    out = []
    S = len(dets)
    for frame in range(frames_n):
        data = [_scene(s, frame, dets[s], 0) for s in range(S)]
        boxes = [torch.arange(dets[s] * 7, dtype=torch.float32).reshape(dets[s], 7) * 0.1 + frame for s in range(S)]
        frames = [None if (s == 1 and frame == 2) else (torch.zeros(0, 4), boxes[s], data[s][2]) for s in range(S)]
        live = [s for s in range(S) if frames[s] is not None]
        monkeypatch.setattr(TR, "crop_center_resample_scenes", lambda *a, **kw: (
            torch.cat([data[s][0] for s in live]), torch.cat([data[s][1] for s in live])))
        out.append(tracker.step(frames, -2.0, dt=dt(frame)))
    return out


def test_tracker_with_motion_model_runs_the_filter_around_the_step(monkeypatch):
    """with a motion model and no bound the gate is the class gate: same ids and costs as without one; the step calls predict
    before the gate and correct after the update, once each, and never the plain gate"""
    from pcreid_b200.models.tracking import MotionModel, ReIDTracker
    calls = []
    _patch(monkeypatch, calls)
    dets = [5, 3, 4]
    plain = ReIDTracker(FakeModel(), num_scenes=3, capacity=8, max_age=1, device="cpu")
    motion = ReIDTracker(FakeModel(), num_scenes=3, capacity=8, max_age=1, device="cpu", motion=MotionModel(gate_chi2=None))
    want = _run(monkeypatch, plain, dets, 4)
    assert "track_predict" not in calls and not hasattr(plain.table, "kf_box")
    calls.clear()
    got = _run(monkeypatch, motion, dets, 4, dt=lambda frame: [0.5, None if frame == 2 else 1.0, 2.0])   # scene 1 frozen
    assert calls == ["track_predict", "track_gate_motion_blocks", "assign", "track_update", "track_correct",
                     "track_scatter"] * 4
    for g, w in zip(got, want):
        for gs, ws in zip(g, w):
            assert (gs is None) == (ws is None)
            if gs is not None:
                assert torch.equal(gs[0], ws[0]) and (ws[1] is None) == (gs[1] is None)
                assert ws[1] is None or torch.equal(gs[1], ws[1])
    for name in ("alive", "track_id", "age", "hits", "box", "count", "next_id", "dropped"):
        assert torch.equal(getattr(plain.table, name), getattr(motion.table, name)), name
    # every alive track of scene 0 was matched or born in the last frame: its estimate lies between the box and the
    # prediction, and a track seen in two frames has picked up the boxes' motion of 1 per frame
    boxes, vel = motion.table.motion(0)
    assert boxes.shape == (int(motion.table.count[0]), 7) and vel.shape == (boxes.shape[0], 3)
    assert bool((vel[:, :3] > 0).any())


def test_tracker_motion_arguments():
    from pcreid_b200.models.tracking import MotionModel, ReIDTracker, TrackTable
    for bad in (dict(init_var=0), dict(init_vel_var=-1), dict(q=-0.1), dict(q_vel=float("nan")), dict(r=0),
                dict(gate_chi2=0), dict(gate_chi2=float("inf"))):
        with pytest.raises(ValueError):
            MotionModel(**bad)
    assert MotionModel(q=0, q_vel=0, gate_chi2=None).gate_chi2 is None
    with pytest.raises(TypeError):
        ReIDTracker(FakeModel(), device="cpu", motion=dict(q=1.0))
    tracker = ReIDTracker(FakeModel(), num_scenes=2, capacity=4, device="cpu", motion=MotionModel())
    frame = (torch.zeros(0, 4), torch.zeros(0, 7), torch.zeros(0, dtype=torch.int64))
    for dt in (-1.0, float("nan"), [1.0], [1.0, float("inf")], [1.0, torch.tensor(1.0)]):
        with pytest.raises((ValueError, TypeError)):
            tracker.step([frame, frame], 0.0, dt=dt)
    with pytest.raises(ValueError):
        TrackTable(1, 4, device="cpu").motion(0)
    tab = _table(2, 3)
    tab.alive[0, 1] = True
    tab.kf_box[0, 1] = 3.0
    tab.kf_vel[0, 1] = 1.0
    box, vel = tab.motion(0)
    assert box.tolist() == [[3.0] * 7] and vel.tolist() == [[1.0] * 3]
    tab.reset(0)
    assert not bool(tab.kf_box[0].any()) and not bool(tab.kf_vel[0].any())


# ---------------------------------------------------------------------------------------------------------- C ABI
@pytest.fixture(scope="module")
def L():
    from pcreid_b200 import _lib
    return _lib.lib()


def test_motion_entry_points_argument_errors_before_any_cuda_call(L):
    nan, inf = float("nan"), float("inf")
    pr = lambda S, C, mA, q=1.0, qv=0.01: L.pcreid_track_predict(S, C, mA, *([None] * 6), q, qv, None)   # noqa: E731
    for a in ((-1, 4, 1), (1, 0, 1), (1, 4, -1), (1, 4, 5), (1, 4, 1, -1.0), (1, 4, 1, nan), (1, 4, 1, 1.0, inf)):
        assert pr(*a) == 1, a
    for a in ((65536, 4, 1), (1, 4097, 1)):
        assert pr(*a) == 3, a
    assert pr(1, 4, 2) == 1                                          # null pointers
    assert pr(0, 4, 2) == 0 and pr(3, 4, 0) == 0 and pr(3, 4, 0, 0.0, 0.0) == 0
    co = lambda S, C, mD, iv=10.0, ivv=1e4, r=1.0: L.pcreid_track_correct(S, C, mD, *([None] * 8), iv, ivv, r, None)  # noqa: E731
    for a in ((-1, 4, 1), (1, 0, 1), (1, 4, -1), (1, 4, 1, 0.0), (1, 4, 1, 10.0, -1.0), (1, 4, 1, 10.0, 1e4, nan),
              (1, 4, 1, inf)):
        assert co(*a) == 1, a
    for a in ((65536, 4, 1), (1, 4097, 1), (1, 4, 4097)):
        assert co(*a) == 3, a
    assert co(2, 4, 3) == 1                                          # null pointers
    assert co(0, 4, 3) == 0 and co(3, 4, 0) == 0

    def gm(S, C, mA, mD, nc=8, r=1.0, chi2=9.21):
        return L.pcreid_track_gate_motion_blocks(S, C, mA, mD, *([None] * 8), nc, 2, 1, None, None, r, chi2, None, None)
    for a in ((-1, 4, 1, 1), (1, 0, 1, 1), (1, 4, -1, 1), (1, 4, 1, -1), (1, 4, 5, 1), (1, 4, 1, 1, -1),
              (1, 4, 1, 1, 8, 0.0), (1, 4, 1, 1, 8, nan, 0.0), (1, 4, 1, 1, 8, 1.0, nan), (1, 4, 1, 1, 8, 1.0, inf)):
        assert gm(*a) == 1, a
    for a in ((65536, 4, 1, 1), (1, 4097, 1, 1), (1, 4, 1, 4097)):
        assert gm(*a) == 3, a
    assert gm(1, 4, 2, 2) == 1 and gm(1, 4, 2, 2, chi2=0.0) == 1        # null pointers
    assert gm(0, 4, 2, 2) == 0 and gm(3, 4, 0, 2) == 0 and gm(3, 4, 2, 0) == 0
