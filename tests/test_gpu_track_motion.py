"""-m gpu: the track table's motion.  pcreid_track_predict / _correct / _gate_motion_blocks against their CPU restatement
(tests/track_motion_reference.py) over random sequences and at the gate's boundaries, bit for bit; ReIDTracker(motion=...)
over many scenes against one-scene trackers; a constant-velocity scene that the filter keeps and the last-box radius splits;
no host synchronisation, opcheck and launch counts."""

import numpy as np
import pytest
import torch

import track_motion_reference as TM
import track_table_reference as TT
from test_gpu_tracker import STATE, _frames, _same_state, pt_model  # noqa: F401  (pt_model: the fixture)

pytestmark = pytest.mark.gpu
DEV = "cuda"
MOTION = ("kf_box", "kf_vel", "kf_cov")


def _tables(S, C):
    from pcreid_b200.models.tracking import TrackTable
    return TrackTable(S, C, device=DEV, motion=True), TrackTable(S, C, device="cpu", motion=True)


def _same_motion(gpu, cpu, what):
    for name in MOTION:
        assert torch.equal(getattr(gpu, name).cpu(), getattr(cpu, name)), (what, name)


# ---------------------------------------------------------------------------------------------------------- kernels
# (S, capacity, largest D_s, max_age)
CASES = [(1, 1, 3, None), (33, 7, 12, 2), (17, 7, 9, 0), (5, 256, 300, 2), (3, 256, 200, None), (2, 4096, 4096, None)]


@pytest.mark.parametrize("case", CASES, ids=[f"S{c[0]}-C{c[1]}-D{c[2]}-age{c[3]}" for c in CASES])
def test_kernels_equal_reference_over_random_sequences(case):
    import pcreid_b200.kernels as K
    S, C, Dmax, max_age = case
    rng = np.random.default_rng(S * 7919 + C + 1)
    gpu, cpu = _tables(S, C)
    r2 = torch.tensor(rng.uniform(0, 30, 8) ** 2, dtype=torch.float32)
    drops = matched = 0
    for step in range(12):
        shapes, tfd = [], []
        for s in range(S):
            if rng.random() < 0.15:                                            # no frame
                shapes.append((0, 0))
                continue
            A = int(cpu.count[s])
            D = int(rng.integers(0, Dmax + 1)) if rng.random() < 0.8 else Dmax
            m = int(rng.integers(0, min(A, D) + 1))
            col = np.full(D, -1, np.int64)
            col[rng.permutation(D)[:m]] = rng.permutation(A)[:m]
            shapes.append((A, D))
            tfd.append(col)
            matched += m
        n = sum(d for _, d in shapes)
        tfd = torch.from_numpy(np.concatenate(tfd) if tfd else np.zeros(0, np.int64))
        label = torch.from_numpy(rng.integers(-1, 4, n).astype(np.int32))
        length = torch.from_numpy(rng.integers(0, 12, n).astype(np.int32))
        box = torch.from_numpy(rng.uniform(-40, 40, (n, 7)).astype(np.float32))
        box[:, 6] = torch.from_numpy(rng.uniform(-8, 8, n).astype(np.float32))     # yaws outside (-pi, pi] too
        dt = [float(np.float32(rng.uniform(0, 2))) if rng.random() < 0.8 else 0.0 for _ in range(S)]
        q, q_vel = (1.0, 0.01) if step % 2 else (0.25, 0.5)
        K.track_predict(gpu, shapes, dt, q, q_vel)
        TM.track_predict(cpu, shapes, dt, q, q_vel)
        _same_motion(gpu, cpu, ("predict", step))
        for radius, chi2 in ((None, None), (r2, 9.21), (None, float(rng.uniform(0.5, 50)))):
            g_gpu = K.track_gate_motion_blocks(gpu, shapes, label.to(DEV), length.to(DEV), box.to(DEV), 8, 2, step % 3 != 0,
                                               None if radius is None else radius.to(DEV), 1.5, chi2)
            g_cpu = TM.track_gate_motion_blocks(cpu, shapes, label, length, box, 8, 2, step % 3 != 0, radius, 1.5, chi2)
            assert torch.equal(g_gpu.cpu(), g_cpu), (step, radius is None, chi2)
        rows_g = torch.cat([gpu.active[s, :a].long() for s, (a, _) in enumerate(shapes)])
        rows_c = torch.cat([cpu.active[s, :a].long() for s, (a, _) in enumerate(shapes)])
        ids_g, det_row_g = K.track_update(gpu, shapes, tfd.to(DEV), label.to(DEV), length.to(DEV), box.to(DEV), max_age)
        ids_c, det_row_c = TT.track_update(cpu, shapes, tfd, label, length, box, max_age)
        assert torch.equal(ids_g.cpu(), ids_c) and torch.equal(det_row_g.cpu(), det_row_c), step
        _same_state(gpu, cpu)
        K.track_correct(gpu, shapes, rows_g, tfd.to(DEV), box.to(DEV), det_row_g, 10.0, 1e4, 1.5)
        TM.track_correct(cpu, shapes, rows_c, tfd, box, det_row_c, 10.0, 1e4, 1.5)
        _same_motion(gpu, cpu, ("correct", step))
        drops = int(cpu.dropped.sum())
    assert matched > 0 and bool(torch.isfinite(cpu.kf_cov).all())
    if C < 4096:
        assert drops > 0


def _one_track(q_box, vel, cov_x, cov_y):
    """one-slot tables, on the device and on the CPU, whose track was born at the origin, given velocity vel, predicted by
    dt = 1 without process noise and then given the position variances cov_x, cov_y; and the detections q_box"""
    import pcreid_b200.kernels as K
    gpu, cpu = _tables(1, 1)
    for t, (update, correct, predict), dev in ((gpu, (K.track_update, K.track_correct, K.track_predict), DEV),
                                               (cpu, (TT.track_update, TM.track_correct, TM.track_predict), "cpu")):
        zero, tfd = torch.zeros((1, 7), device=dev), torch.tensor([-1], device=dev)
        _, rows = update(t, [(0, 1)], tfd, torch.zeros(1, dtype=torch.int32, device=dev),
                         torch.full((1,), 5, dtype=torch.int32, device=dev), zero)
        correct(t, [(0, 1)], torch.zeros(0, dtype=torch.long, device=dev), tfd, zero, rows)
        t.kf_vel[0, 0] = torch.tensor(vel)
        predict(t, [(1, 0)], 1.0, 0.0, 0.0)
        t.kf_cov[0, 0, 0], t.kf_cov[0, 0, 3] = cov_x, cov_y
    q = torch.tensor(q_box, dtype=torch.float32).reshape(-1, 7)
    n = q.shape[0]
    return gpu, cpu, (torch.zeros(n, dtype=torch.int32), torch.full((n,), 5, dtype=torch.int32), q)


def test_gate_boundaries():
    import pcreid_b200.kernels as K
    # predicted centre (3, 4); Sx = 3, Sy = 5 with r = 1
    gpu, cpu, dets = _one_track([[3.0, 4.0] + [0.0] * 5, [0.0] * 7, [6.0, 4.0] + [0.0] * 5, [6.0, 9.0] + [0.0] * 5],
                                [3.0, 4.0, 0.0], 2.0, 4.0)
    assert gpu.kf_box[0, 0, :2].tolist() == [3.0, 4.0]
    dg = [t.to(DEV) for t in dets]
    r2 = torch.full((8,), 25.0)

    def both(**kw):
        g = K.track_gate_motion_blocks(gpu, [(1, 4)], *dg, **{k: (v.to(DEV) if isinstance(v, torch.Tensor) else v)
                                                               for k, v in kw.items()}).cpu()
        c = TM.track_gate_motion_blocks(cpu, [(1, 4)], *dets, **kw)
        assert torch.equal(g, c), kw
        return g.tolist()
    # the radius is measured from the predicted centre, exactly at it passes; (6, 4) is 3 m from the prediction and 7.2 m
    # from the last matched box (the origin)
    assert both(radius_sq=r2) == [True, True, True, False]
    assert both(radius_sq=torch.full((8,), 24.99)) == [True, False, True, False]
    # d^2 = 0, 9/3 + 16/5, 3, 3 + 25/5 = 8: exactly the bound passes
    assert both(r=1.0, gate_chi2=8.0) == [True] * 4
    assert both(r=1.0, gate_chi2=7.999) == [True, True, True, False]
    assert both(r=1.0, gate_chi2=3.0) == [True, False, True, False]
    assert both(radius_sq=r2, r=1.0, gate_chi2=3.0) == [True, False, True, False]
    # a bound equal to one pair's float32 distance
    rng = np.random.default_rng(5)
    q = torch.from_numpy(rng.uniform(-6, 12, (64, 7)).astype(np.float32))
    gpu, cpu, dets = _one_track(q.tolist(), [1.5, -2.0, 0.0], 0.7, 1.3)
    dx, dy = cpu.kf_box[0, 0, 0] - q[:, 0], cpu.kf_box[0, 0, 1] - q[:, 1]
    d2 = dx * dx / (cpu.kf_cov[0, 0, 0] + 1.0) + dy * dy / (cpu.kf_cov[0, 0, 3] + 1.0)
    chi2 = float(d2[17])
    g = K.track_gate_motion_blocks(gpu, [(1, 64)], *[t.to(DEV) for t in dets], r=1.0, gate_chi2=chi2).cpu()
    assert torch.equal(g, TM.track_gate_motion_blocks(cpu, [(1, 64)], *dets, r=1.0, gate_chi2=chi2)) and bool(g[17])
    assert torch.equal(g, d2 <= chi2) and 0 < int(g.sum()) < 64


def _kernel_args():
    import pcreid_b200.kernels as K
    gpu, _ = _tables(3, 8)
    shapes = [(0, 3), (0, 0), (0, 2)]
    lab = torch.tensor([1, 2, 1, 1, 3], dtype=torch.int32, device=DEV)
    ln = torch.full((5,), 4, dtype=torch.int32, device=DEV)
    bx = torch.randn((5, 7), device=DEV)
    tfd = torch.full((5,), -1, device=DEV)
    _, det_row = K.track_update(gpu, shapes, tfd, lab, ln, bx)
    K.track_correct(gpu, shapes, torch.zeros(0, dtype=torch.long, device=DEV), tfd, bx, det_row)
    return gpu, [(3, 3), (0, 0), (2, 2)], lab, ln, bx


def test_no_host_synchronisation_and_opcheck():
    import pcreid_b200.kernels as K
    gpu, shapes, lab, ln, bx = _kernel_args()
    tfd = torch.tensor([1, -1, 0, -1, 1], device=DEV)
    r2 = torch.full((8,), 4.0, device=DEV)
    K.track_predict(gpu, shapes, [0.5, 1.0, 2.0])                              # warm-up: pinned buffers
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        rows = torch.cat([gpu.active[s, :a].long() for s, (a, _) in enumerate(shapes)])
        K.track_predict(gpu, shapes, [0.5, 1.0, 2.0])
        gate = K.track_gate_motion_blocks(gpu, shapes, lab, ln, bx, radius_sq=r2, gate_chi2=9.21)
        _, det_row = K.track_update(gpu, shapes, tfd, lab, ln, bx, max_age=2)
        K.track_correct(gpu, shapes, rows, tfd, bx, det_row)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert gate.shape == (13,)
    off = torch.tensor([[0, 3, 3, 5], [0, 3, 3, 5], [0, 9, 9, 13]], dtype=torch.int64, device=DEV)
    dt = torch.tensor([0.5, 1.0, 2.0], device=DEV)
    ops = torch.ops.pcreid
    torch.library.opcheck(ops.track_predict, (3, 8, 3, off, gpu.active, dt, gpu.kf_box.clone(), gpu.kf_vel.clone(),
                                              gpu.kf_cov.clone(), 1.0, 0.01), test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(ops.track_correct, (3, 8, 3, off, rows, tfd, bx, det_row, gpu.kf_box.clone(), gpu.kf_vel.clone(),
                                              gpu.kf_cov.clone(), 10.0, 1e4, 1.0), test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(ops.track_gate_motion_blocks, (3, 8, 3, 3, off, gpu.active, gpu.label, gpu.length, gpu.kf_box, lab, ln,
                                                         bx, 8, 2, 1, r2, gpu.kf_cov, 1.0, 9.21,
                                                         torch.empty(13, dtype=torch.bool, device=DEV)),
                          test_utils=("test_schema", "test_faketensor"))


def test_wrapper_argument_checks():
    import pcreid_b200.kernels as K
    from pcreid_b200.models.tracking import TrackTable
    gpu, shapes, lab, ln, bx = _kernel_args()
    plain = TrackTable(3, 8, device=DEV)
    with pytest.raises(ValueError):
        K.track_predict(plain, shapes, 1.0)                                    # no motion state
    with pytest.raises(ValueError):
        K.track_predict(gpu, shapes, [1.0, 2.0])                               # one dt per scene
    with pytest.raises(ValueError):
        K.track_predict(gpu, shapes, -1.0)
    with pytest.raises(TypeError):
        K.track_predict(gpu, shapes, torch.ones(3, device=DEV))
    with pytest.raises(ValueError):
        K.track_gate_motion_blocks(gpu, shapes, lab, ln, bx, gate_chi2=0.0)
    tfd = torch.full((5,), -1, device=DEV)
    with pytest.raises(ValueError):
        K.track_correct(gpu, shapes, torch.zeros(4, dtype=torch.long, device=DEV), tfd, bx,
                        torch.zeros(5, dtype=torch.int32, device=DEV))            # track_rows holds sum A_s = 5 rows
    with pytest.raises(ValueError):
        K.track_correct(gpu, shapes, torch.zeros(5, dtype=torch.long, device=DEV), tfd, bx,
                        torch.zeros(5, dtype=torch.int32, device=DEV), r=0.0)


# ---------------------------------------------------------------------------------------------------------- ReIDTracker
def test_many_scenes_equal_one_scene_trackers(pt_model):
    """17 scenes in one motion tracker against 17 one-scene motion trackers with per-scene dt, a frozen scene, retirement,
    drops and a distance gate: results, costs and every table array including the motion state, bit for bit"""
    from pcreid_b200.models.tracking import MotionModel, ReIDTracker
    pt_model.set_mode("parity_tc")
    rng = np.random.default_rng(23)
    S, C = 17, 12
    sizes = [(int(rng.integers(0, 30000)), int(rng.integers(0, 14))) for _ in range(S)]
    kw = dict(capacity=C, max_age=2, max_distance=[60.0, 45.0, 80.0, 1.0, 1.0, 1.0, 1.0, 1.0], motion=MotionModel(q_vel=0.5))
    multi = ReIDTracker(pt_model, num_scenes=S, **kw)
    single = [ReIDTracker(pt_model, num_scenes=1, **kw) for _ in range(S)]
    matched = 0
    try:
        for frame in range(6):
            frames, ranks = _frames(sizes, frame, 29, none_scene=2)
            dt = [float(rng.choice([0.0, 0.1, 0.5, 1.0])) for _ in range(S)]
            got = multi.step(frames, -2.0, sample_ranks=ranks, dt=dt)
            for s in range(S):
                known = int(single[s].table.next_id[0])
                want = single[s].step([frames[s]], -2.0, sample_ranks=[ranks[s]], dt=dt[s])[0]
                if frames[s] is None:
                    assert got[s] is None and want is None
                    continue
                assert torch.equal(got[s][0], want[0]), (frame, s)
                assert (got[s][1] is None) == (want[1] is None) and (want[1] is None or torch.equal(got[s][1], want[1]))
                matched += int(((want[0] >= 0) & (want[0] < known)).sum())
                a, b = multi.table, single[s].table
                for name in STATE + MOTION:
                    x, y = getattr(a, name)[s], getattr(b, name)[0]
                    if name == "active":                                # global rows; entries past the count are stale
                        n = int(b.count[0])
                        x, y = x[:n] - s * C, y[:n]
                    assert torch.equal(x, y), (frame, s, name)
    finally:
        pt_model.set_mode("parity")
    assert matched > 0 and int(multi.table.dropped.sum()) > 0 and not bool(multi.table.alive.all())


def _moving_scene(n_obj, frame, step=3.0, gap=50.0, pts_per_obj=300, seed=0):
    """n_obj boxes (4 x 2 x 1.5 m) gap metres apart in y, all moving step metres per frame in x, and a sweep with points in
    every box"""
    g = torch.Generator().manual_seed(seed + frame)
    boxes = torch.zeros(n_obj, 7)
    boxes[:, 0] = 10.0 + step * frame
    boxes[:, 1] = gap * torch.arange(n_obj, dtype=torch.float32)
    boxes[:, 3:6] = torch.tensor([4.0, 2.0, 1.5])
    local = (torch.rand(n_obj, pts_per_obj, 3, generator=g) - 0.5) * torch.tensor([3.6, 1.6, 1.2])
    pts = (local + boxes[:, None, :3]).reshape(-1, 3)
    sweep = torch.cat([pts, torch.zeros(pts.shape[0], 1)], 1)
    return sweep.to(DEV), boxes.to(DEV), torch.zeros(n_obj, dtype=torch.int64, device=DEV)


def test_constant_velocity_objects_keep_their_ids(pt_model, monkeypatch):
    """objects 50 m apart moving 3 m per step: with MotionModel(init_vel_var=25) every object keeps its birth id for 10 steps
    and its velocity estimate ends within 0.1 m/step of the truth; a radius of 1.5 m around the last box splits them into new
    ids every step"""
    import pcreid_b200.kernels as K
    from pcreid_b200.models.tracking import MotionModel, ReIDTracker
    n_obj, steps = 6, 10
    d2 = []
    real_gate = K.track_gate_motion_blocks

    def gate(table, shapes, det_label, det_length, det_box, *a, **kw):
        # the Mahalanobis distance of every pair on the predicted state the kernel gates on (read back: test only)
        A = shapes[0][0]
        if A == 0:
            return real_gate(table, shapes, det_label, det_length, det_box, *a, **kw)
        rows = table.active[0, :A].long()
        p, P = table.kf_box.view(-1, 7)[rows, :2], table.kf_cov.view(-1, 13)[rows][:, [0, 3]] + 1.0
        d = p[:, None, :] - det_box[None, :, :2]
        d2.append(((d * d) / P[:, None, :]).sum(-1).cpu())
        return real_gate(table, shapes, det_label, det_length, det_box, *a, **kw)
    monkeypatch.setattr(K, "track_gate_motion_blocks", gate)
    common = dict(num_scenes=1, capacity=64, use_lengths=False)
    tracker = ReIDTracker(pt_model, motion=MotionModel(init_vel_var=25.0), **common)
    plain = ReIDTracker(pt_model, max_distance=1.5, **common)
    ids, ids_plain = [], []
    for frame in range(steps):
        sweep, boxes, labels = _moving_scene(n_obj, frame)
        ids.append(tracker.step([(sweep, boxes, labels)], -1e6, dt=1.0)[0][0].tolist())
        ids_plain.append(plain.step([(sweep, boxes, labels)], -1e6)[0][0].tolist())
    assert all(x == list(range(n_obj)) for x in ids), ids
    _, vel = tracker.table.motion(0)
    # measured on a B200 (1000 W): vx = 2.984377 for every object after the nine corrections; a float64 run of one axis of
    # this filter on the host gives 2.984
    assert float((vel[:, 0] - 3.0).abs().max()) < 0.1 and float(vel[:, 1:].abs().max()) < 0.1
    own = max(float(m.diagonal().max()) for m in d2)
    neighbour = min(float((m + torch.eye(n_obj) * 1e9).min()) for m in d2)
    # measured on a B200 (1000 W): largest own d^2 0.2432, smallest neighbour d^2 67.81, against the bound 9.21 (the host
    # float64 calculation gives <= 0.25 and >= 59.7)
    assert own <= 0.25 and neighbour >= 59.7
    for frame in range(1, steps):
        assert all(i >= n_obj * frame for i in ids_plain[frame]), ids_plain     # every object got a new id
    assert sorted(ids_plain[-1]) == list(range(n_obj * (steps - 1), n_obj * steps))


def test_launches_do_not_grow_with_scene_count(pt_model, monkeypatch):
    """with a motion model: predict, the motion gate and correct run once per step for 1 and for 17 scenes, alongside the
    update and scatter; the plain gate never runs"""
    from pcreid_b200 import torch_ops
    import pcreid_b200.kernels as K
    import pcreid_b200.models.tracking as TR
    counted = ("track_predict", "track_correct", "track_gate_motion_blocks", "track_gate_blocks", "track_update",
               "track_scatter", "lsap_blocks")
    calls = {}

    class Counting:
        def __getattr__(self, name):
            op = getattr(torch_ops.ops, name)
            if name not in counted:
                return op

            def wrapped(*a, **kw):
                calls[name] = calls.get(name, 0) + 1
                return op(*a, **kw)
            return wrapped

    monkeypatch.setattr(K, "_OPS", Counting())
    pt_model.set_mode("parity_tc")
    per_S = {}
    try:
        for S in (1, 17):
            rng = np.random.default_rng(S)
            sizes = [(int(rng.integers(1000, 20000)), int(rng.integers(2, 10))) for _ in range(S)]
            tracker = TR.ReIDTracker(pt_model, num_scenes=S, capacity=64, motion=TR.MotionModel())
            frames, ranks = _frames(sizes, 0, 77)
            tracker.step(frames, -2.0, sample_ranks=ranks)
            frames, ranks = _frames(sizes, 2, 77)
            calls.clear()
            tracker.step(frames, -2.0, sample_ranks=ranks, dt=[0.1] * S)
            per_S[S] = dict(calls)
    finally:
        pt_model.set_mode("parity")
    for S in (1, 17):
        c = per_S[S]
        for k in ("track_predict", "track_correct", "track_gate_motion_blocks", "track_update", "track_scatter", "lsap_blocks"):
            assert c.get(k) == 1, (S, k, c)
        assert "track_gate_blocks" not in c, c
