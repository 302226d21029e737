"""-m gpu: the device track table.  pcreid_track_gate_blocks / _update / _scatter against their plain-torch restatement
(tests/track_table_reference.py) over random sequences, the gate against class_gate and the float32 distance rule, no host
synchronisation, opcheck, and ReIDTracker against PointReidentifier.step and against one-scene trackers -- all bit for bit --
plus launch counts that do not grow with the scene count."""

import numpy as np
import pytest
import torch

import helpers
import track_table_reference as TT
from test_gpu_multiscene import _ranks, _scenes

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module")
def pt_model():
    m, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    return m


def _tables(S, C, replace_all=False):
    from pcreid_b200.models.tracking import TrackTable
    return TrackTable(S, C, replace_all, device=DEV), TrackTable(S, C, replace_all, device="cpu")


STATE = ("alive", "track_id", "label", "length", "age", "hits", "box", "active", "next_id", "dropped", "count")


def _same_state(gpu, cpu):
    for name in STATE:
        assert torch.equal(getattr(gpu, name).cpu(), getattr(cpu, name)), name


# ---------------------------------------------------------------------------------------------------------- kernels
# (S, capacity, largest D_s, max_age, replace_all, feature row (shape, dtype))
CASES = [(1, 1, 3, None, False, ((5,), torch.float16)),
         (33, 7, 12, 2, True, ((3, 8), torch.float32)),
         (17, 7, 9, 0, False, ((6,), torch.uint8)),
         (5, 256, 300, 2, False, ((64, 8), torch.float32)),
         (3, 256, 200, None, True, ((7,), torch.int64)),
         (2, 4096, 4096, None, False, ((4,), torch.float32)),
         (2, 4096, 4096, 0, True, ((3,), torch.float16))]


@pytest.mark.parametrize("case", CASES, ids=[f"S{c[0]}-C{c[1]}-D{c[2]}-age{c[3]}-ra{int(c[4])}" for c in CASES])
def test_kernels_equal_reference_over_random_sequences(case):
    import pcreid_b200.kernels as K
    S, C, Dmax, max_age, replace_all, (frow, fdtype) = case
    rng = np.random.default_rng(S * 7919 + C)
    gpu, cpu = _tables(S, C, replace_all)
    N = 4
    for t in (gpu, cpu):
        t.xyz = torch.zeros((S * C, N, 3), device=t.device)
        t.feat = torch.zeros((S * C,) + frow, dtype=fdtype, device=t.device)
    r2 = torch.tensor(rng.uniform(0, 30, 8) ** 2, dtype=torch.float32)
    drops = 0
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
        n = sum(d for _, d in shapes)
        tfd = torch.from_numpy(np.concatenate(tfd) if tfd else np.zeros(0, np.int64))
        label = torch.from_numpy(rng.integers(-1, 10, n).astype(np.int32))
        length = torch.from_numpy(rng.integers(0, 12, n).astype(np.int32))
        box = torch.from_numpy(rng.uniform(-40, 40, (n, 7)).astype(np.float32))
        xyz = torch.randn(n, N, 3, generator=torch.Generator().manual_seed(step))
        feat = torch.from_numpy(rng.integers(0, 100, (n,) + frow)).to(fdtype)
        for radius in (None, r2):
            g_gpu = K.track_gate_blocks(gpu, shapes, label.to(DEV), length.to(DEV), box.to(DEV), 8, 2, step % 3 != 0,
                                        None if radius is None else radius.to(DEV))
            g_cpu = TT.track_gate_blocks(cpu, shapes, label, length, box, 8, 2, step % 3 != 0, radius)
            assert torch.equal(g_gpu.cpu(), g_cpu), (step, radius is None)
        ids_g, rows_g = K.track_update(gpu, shapes, tfd.to(DEV), label.to(DEV), length.to(DEV), box.to(DEV), max_age,
                                       replace_all)
        ids_c, rows_c = TT.track_update(cpu, shapes, tfd, label, length, box, max_age, replace_all)
        assert torch.equal(ids_g.cpu(), ids_c) and torch.equal(rows_g.cpu(), rows_c), step
        _same_state(gpu, cpu)
        K.track_scatter(rows_g, xyz.to(DEV), feat.to(DEV), gpu.xyz, gpu.feat)
        TT.track_scatter(rows_c, xyz, feat, cpu.xyz, cpu.feat)
        assert torch.equal(gpu.xyz.cpu(), cpu.xyz) and torch.equal(gpu.feat.cpu(), cpu.feat), step
        drops = int(cpu.dropped.sum())
    if not (C == 4096 and max_age == 0):                  # there every unmatched detection finds a slot
        assert drops > 0


def test_gate_equals_class_gate_and_distance_rule():
    import pcreid_b200.kernels as K
    from pcreid_b200.models.tracking import class_gate
    rng = np.random.default_rng(3)
    S, C = 6, 64
    gpu, cpu = _tables(S, C)
    # fill the tables with tracks of random labels, lengths and integer-valued boxes
    D = [int(rng.integers(0, 40)) for _ in range(S)]
    n = sum(D)
    lab = torch.from_numpy(rng.integers(-1, 10, n).astype(np.int32))
    ln = torch.from_numpy(rng.integers(0, 6, n).astype(np.int32))
    bx = torch.from_numpy(rng.integers(-6, 7, (n, 7)).astype(np.float32))
    shapes = [(0, d) for d in D]
    K.track_update(gpu, shapes, torch.full((n,), -1, device=DEV), lab.to(DEV), ln.to(DEV), bx.to(DEV))
    TT.track_update(cpu, shapes, torch.full((n,), -1), lab, ln, bx)
    _same_state(gpu, cpu)
    Dd = [int(rng.integers(0, 50)) for _ in range(S)]
    m = sum(Dd)
    dl = torch.from_numpy(rng.integers(-1, 10, m).astype(np.int32))
    dn = torch.from_numpy(rng.integers(0, 6, m).astype(np.int32))
    db = torch.from_numpy(rng.integers(-6, 7, (m, 7)).astype(np.float32))
    shapes = [(int(cpu.count[s]), Dd[s]) for s in range(S)]
    for use_lengths in (True, False):
        for nc, mp in ((8, 2), (5, 4)):
            got = K.track_gate_blocks(gpu, shapes, dl.to(DEV), dn.to(DEV), db.to(DEV), nc, mp, use_lengths).cpu()
            want, d0 = [], 0
            for s, (A, Ds) in enumerate(shapes):
                want.append(class_gate(dl[d0:d0 + Ds].long(), cpu.label[s, :A].long(), dn[d0:d0 + Ds].long(),
                                       cpu.length[s, :A].long(), use_lengths, nc, mp).reshape(-1))
                d0 += Ds
            assert torch.equal(got, torch.cat(want)), (use_lengths, nc, mp)
    # integer boxes: many pairs at exactly the radius (3-4-5, 0-5, ...); and radii equal to one pair's f32 distance
    for r2 in (torch.full((8,), 25.0), torch.tensor([0.0, 1.0, 25.0, 50.0, 100.0, 2.0, 400.0, 1e9])):
        got = K.track_gate_blocks(gpu, shapes, dl.to(DEV), dn.to(DEV), db.to(DEV), 8, 2, True, r2.to(DEV)).cpu()
        want = TT.track_gate_blocks(cpu, shapes, dl, dn, db, 8, 2, True, r2)
        assert torch.equal(got, want)
        plain = TT.track_gate_blocks(cpu, shapes, dl, dn, db, 8, 2, True)
        assert 0 < int(want.sum()) < int(plain.sum())
    fbx = torch.from_numpy(rng.uniform(-6, 6, (m, 7)).astype(np.float32))
    i = int(torch.nonzero(plain)[0])
    s = next(k for k in range(S) if sum(a * d for a, d in shapes[:k + 1]) > i)
    e = i - sum(a * d for a, d in shapes[:s])
    t, dj = divmod(e, shapes[s][1])
    row, dj = int(cpu.active[s, t]), sum(d for _, d in shapes[:s]) + dj
    dx, dy = cpu.box.view(-1, 7)[row, 0] - fbx[dj, 0], cpu.box.view(-1, 7)[row, 1] - fbx[dj, 1]
    r2 = torch.full((8,), float(dx * dx + dy * dy), dtype=torch.float32)
    got = K.track_gate_blocks(gpu, shapes, dl.to(DEV), dn.to(DEV), fbx.to(DEV), 8, 2, True, r2.to(DEV)).cpu()
    want = TT.track_gate_blocks(cpu, shapes, dl, dn, fbx, 8, 2, True, r2)
    assert torch.equal(got, want) and bool(want[i])


def _kernel_args():
    import pcreid_b200.kernels as K
    gpu, _ = _tables(3, 8)
    gpu.xyz, gpu.feat = torch.zeros((24, 4, 3), device=DEV), torch.zeros((24, 5), device=DEV)
    shapes = [(0, 3), (0, 0), (0, 2)]
    lab = torch.tensor([1, 2, 1, 1, 3], dtype=torch.int32, device=DEV)
    ln = torch.full((5,), 4, dtype=torch.int32, device=DEV)
    bx = torch.zeros((5, 7), device=DEV)
    ids, rows = K.track_update(gpu, shapes, torch.full((5,), -1, device=DEV), lab, ln, bx)
    return gpu, [(3, 3), (0, 0), (2, 2)], lab, ln, bx, rows


def test_no_host_synchronisation_and_opcheck():
    import pcreid_b200.kernels as K
    gpu, shapes, lab, ln, bx, rows = _kernel_args()
    tfd = torch.tensor([1, -1, 0, -1, 1], device=DEV)
    xyz, feat = torch.randn(5, 4, 3, device=DEV), torch.randn(5, 5, device=DEV)
    r2 = torch.full((8,), 4.0, device=DEV)
    K.track_gate_blocks(gpu, shapes, lab, ln, bx, radius_sq=r2)                  # warm-up: pinned buffers
    K.track_scatter(rows, xyz, feat, gpu.xyz, gpu.feat)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        gate = K.track_gate_blocks(gpu, shapes, lab, ln, bx, radius_sq=r2)
        ids, rows = K.track_update(gpu, shapes, tfd, lab, ln, bx, max_age=2)
        K.track_scatter(rows, xyz, feat, gpu.xyz, gpu.feat)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert gate.shape == (13,) and ids.shape == (5,)
    off = torch.tensor([[0, 3, 3, 5], [0, 3, 3, 5], [0, 9, 9, 13]], dtype=torch.int64, device=DEV)
    ops = torch.ops.pcreid
    torch.library.opcheck(ops.track_gate_blocks, (3, 8, 3, 3, off, gpu.active, gpu.label, gpu.length, gpu.box, lab, ln, bx, 8, 2,
                                                  1, r2, torch.empty(13, dtype=torch.bool, device=DEV)),
                          test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(ops.track_update, (3, 8, 3, off, torch.full((5,), -1, device=DEV), lab, ln, bx, 1, 0,
                                             gpu.alive.clone(), gpu.track_id.clone(), gpu.label.clone(), gpu.length.clone(),
                                             gpu.age.clone(), gpu.hits.clone(), gpu.box.clone(), gpu.next_id.clone(),
                                             gpu.dropped.clone(), gpu.active.clone(), gpu.count.clone(),
                                             torch.empty(5, dtype=torch.int64, device=DEV),
                                             torch.empty(5, dtype=torch.int32, device=DEV)),
                          test_utils=("test_schema", "test_faketensor"))
    torch.library.opcheck(ops.track_scatter, (5, rows, 48, xyz, gpu.xyz.clone(), 20, feat, gpu.feat.clone()),
                          test_utils=("test_schema", "test_faketensor"))


def test_wrapper_argument_checks():
    import pcreid_b200.kernels as K
    gpu, shapes, lab, ln, bx, rows = _kernel_args()
    with pytest.raises(ValueError):
        K.track_gate_blocks(gpu, shapes[:2], lab, ln, bx)                        # one shape per scene
    with pytest.raises(ValueError):
        K.track_gate_blocks(gpu, [(9, 3), (0, 0), (0, 2)], lab, ln, bx)         # A_s > capacity
    with pytest.raises(ValueError):
        K.track_gate_blocks(gpu, shapes, lab.long(), ln, bx)                     # labels must be int32
    with pytest.raises(ValueError):
        K.track_update(gpu, shapes, torch.zeros(4, dtype=torch.int64, device=DEV), lab, ln, bx)
    with pytest.raises(ValueError):
        K.track_update(gpu, shapes, torch.zeros(5, dtype=torch.int64, device=DEV), lab, ln, bx, max_age=-1)
    with pytest.raises(ValueError):
        K.track_scatter(rows, torch.zeros(5, 4, 3, device=DEV), torch.zeros(5, 6, device=DEV), gpu.xyz, gpu.feat)


# ---------------------------------------------------------------------------------------------------------- ReIDTracker
def _frames(sizes, frame, seed, none_scene=None):
    sc = _scenes([(P, B) for P, B in sizes], seed + 1000 * frame)
    frames, ranks = [], []
    for s, (pts, boxes) in enumerate(sc):
        B = boxes.shape[0]
        dl = torch.arange(B, device=DEV) % 3
        if B:
            dl[-1] = 9                                                          # never compared
        none = s == none_scene and frame == 1
        frames.append(None if none else (pts, boxes, dl))
        ranks.append(None if none else _ranks(B, 128, 31 * s + frame))
    return frames, ranks


@pytest.mark.parametrize("kind,mode", [("pt", "parity_tc"), ("pt", "fast"), ("concat", "parity")])
@pytest.mark.parametrize("replace_all", [False, True])
def test_tracker_equals_point_reidentifier_step(pt_model, kind, mode, replace_all):
    """ReIDTracker(num_scenes=1) against PointReidentifier.step with track_index = arange(len(bank)): costs, assignments (a
    detection's id is its bank row) and bank rows"""
    from pcreid_b200.models.tracking import PointFeatureSet, PointReidentifier, ReIDTracker
    model = pt_model if kind == "pt" else helpers.build_pair("concat", (128, 64, 32), device=DEV)[0]
    model.set_mode(mode)
    C = 256
    tracker = ReIDTracker(model, num_scenes=1, capacity=C, replace_all=replace_all)
    bank = PointFeatureSet(replace_all)
    labels = torch.zeros(0, dtype=torch.int64, device=DEV)
    matched = 0
    try:
        for frame in range(5):
            frames, ranks = _frames([(20000, 9 + frame)], frame, 0)
            (ids, cost), = tracker.step(frames, -2.0, sample_ranks=ranks)
            ref = PointReidentifier(model, bank)
            tfd, new_rows, want_cost = ref.step(*frames[0], torch.arange(len(bank), device=DEV), labels, -2.0,
                                                sample_rank=ranks[0])
            want = tfd.clone()
            want[tfd < 0] = new_rows
            assert torch.equal(ids, want), (mode, frame)
            assert (cost is None) == (want_cost is None) and (cost is None or torch.equal(cost, want_cost)), (mode, frame)
            labels = torch.cat([labels, frames[0][2][tfd < 0]])
            n = len(bank)
            tab = tracker.table
            assert torch.equal(tab.xyz[:n], bank.pts_xyz) and torch.equal(tab.feat[:n], bank.pts_feats)
            assert torch.equal(tab.length[0, :n].long(), bank.lengths) and torch.equal(tab.label[0, :n].long(), labels)
            assert int(tab.count[0]) == n and torch.equal(tab.track_id[0, :n], torch.arange(n, device=DEV))
            matched += int((tfd >= 0).sum())
    finally:
        model.set_mode("parity")
    assert matched > 0


def test_many_scenes_equal_one_scene_trackers(pt_model):
    """S scenes in one ReIDTracker against S one-scene ReIDTrackers with retirement, a small capacity (drops) and a
    per-class centre-distance gate: results, costs and every table array, bit for bit"""
    from pcreid_b200.models.tracking import ReIDTracker
    pt_model.set_mode("parity_tc")
    rng = np.random.default_rng(17)
    S, C = 17, 12
    sizes = [(int(rng.integers(0, 30000)), int(rng.integers(0, 14))) for _ in range(S)]
    kw = dict(capacity=C, max_age=2, max_distance=[30.0, 25.0, 40.0, 1.0, 1.0, 1.0, 1.0, 1.0])
    multi = ReIDTracker(pt_model, num_scenes=S, **kw)
    single = [ReIDTracker(pt_model, num_scenes=1, **kw) for _ in range(S)]
    matched = 0
    try:
        for frame in range(6):
            frames, ranks = _frames(sizes, frame, 17, none_scene=2)
            got = multi.step(frames, -2.0, sample_ranks=ranks)
            for s in range(S):
                want = single[s].step([frames[s]], -2.0, sample_ranks=[ranks[s]])[0]
                if frames[s] is None:
                    assert got[s] is None and want is None
                    continue
                assert torch.equal(got[s][0], want[0]), (frame, s)
                assert (got[s][1] is None) == (want[1] is None) and (want[1] is None or torch.equal(got[s][1], want[1]))
                matched += int((want[0] >= 0).sum())
                a, b = multi.table, single[s].table
                for name in STATE:
                    x, y = getattr(a, name)[s], getattr(b, name)[0]
                    if name == "active":                                # global rows; entries past the count are stale
                        n = int(b.count[0])
                        x, y = x[:n] - s * C, y[:n]
                    assert torch.equal(x, y), (frame, s, name)
                rows = slice(s * C, (s + 1) * C)
                alive = b.alive[0]
                assert torch.equal(a.xyz[rows][alive], b.xyz[alive]) and torch.equal(a.feat[rows][alive], b.feat[alive])
    finally:
        pt_model.set_mode("parity")
    assert matched > 0 and int(multi.table.dropped.sum()) > 0 and not bool(multi.table.alive.all())


def test_launches_do_not_grow_with_scene_count(pt_model, monkeypatch):
    """the table's gate, update and scatter, the crop passes and lsap run once per step for 1 and for 17 scenes; the bank
    methods of PointFeatureSet and class_gate are never called"""
    from pcreid_b200 import torch_ops
    from pcreid_b200.models import frontend
    import pcreid_b200.kernels as K
    import pcreid_b200.models.tracking as TR
    counted = ("crop_mask_scenes", "crop_gather_scenes", "lsap_blocks", "track_gate_blocks", "track_update", "track_scatter",
               "pair_p1a2", "pair_p1b_n", "pair_p2y", "crop_mask", "crop_gather", "lsap")
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

    def never(*a, **kw):
        raise AssertionError("the track table's step must not use the per-scene bank or gate")

    monkeypatch.setattr(frontend, "_OPS", Counting())
    monkeypatch.setattr(K, "_OPS", Counting())
    from pcreid_b200.models import fused_pairs
    if hasattr(fused_pairs, "_OPS"):
        monkeypatch.setattr(fused_pairs, "_OPS", Counting())
    for name in ("replace_old", "store_new"):
        monkeypatch.setattr(TR.PointFeatureSet, name, never)
    monkeypatch.setattr(TR, "class_gate", never)
    pt_model.set_mode("parity_tc")
    per_S = {}
    try:
        for S in (1, 17):
            rng = np.random.default_rng(S)
            sizes = [(int(rng.integers(1000, 20000)), int(rng.integers(2, 10))) for _ in range(S)]
            tracker = TR.ReIDTracker(pt_model, num_scenes=S, capacity=64)
            frames, ranks = _frames(sizes, 0, 77)
            tracker.step(frames, -2.0, sample_ranks=ranks)                       # first frame: tracks to match against
            frames, ranks = _frames(sizes, 2, 77)
            calls.clear()
            tracker.step(frames, -2.0, sample_ranks=ranks)
            per_S[S] = dict(calls)
    finally:
        pt_model.set_mode("parity")
    for S in (1, 17):
        c = per_S[S]
        for k in ("crop_mask_scenes", "crop_gather_scenes", "lsap_blocks", "track_gate_blocks", "track_update", "track_scatter"):
            assert c.get(k) == 1, (S, k, c)
        assert "lsap" not in c and "crop_mask" not in c and "crop_gather" not in c, c
    fused = ("pair_p1a2", "pair_p1b_n", "pair_p2y")
    assert sum(per_S[1].get(k, 0) for k in fused) > 0
    assert all(per_S[17].get(k, 0) == per_S[1].get(k, 0) for k in fused), per_S
