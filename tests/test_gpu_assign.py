"""-m gpu: the gated linear assignment kernel (csrc/assign.cu, kernels.linear_assignment) against the scipy oracle
(tests/assign_reference.py), and PointReidentifier.step against the same steps composed by hand."""
import copy

import numpy as np
import pytest
import torch

import assign_reference as R
import helpers
from oracle import reid_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _mask(kind, T, D, rng):
    if kind == "none":
        return None
    if kind == "half":
        return rng.random((T, D)) < 0.5
    lt, ld = rng.integers(0, 8, T), rng.integers(0, 8, D)              # 8-class gate
    return lt[:, None] == ld[None, :]


def _solve(S, tau, mask=None):
    from pcreid_b200.kernels import linear_assignment
    m = None if mask is None else torch.from_numpy(mask).to(DEV)
    d4t, t4d = linear_assignment(torch.from_numpy(S).to(DEV), tau, m)
    assert d4t.dtype == torch.int64 and t4d.dtype == torch.int64 and d4t.is_cuda
    return d4t.cpu().numpy(), t4d.cpu().numpy()


def _check_equal_to_oracle(S, mask, q):
    tau = float(np.float32(np.percentile(S, q)))
    d4t, t4d = _solve(S, tau, mask)
    rd, rt = R.assign(S, tau, mask)
    assert np.array_equal(d4t, rd) and np.array_equal(t4d, rt)


@pytest.mark.parametrize("q", [10, 90])
@pytest.mark.parametrize("mask_kind", ["none", "half", "class8"])
@pytest.mark.parametrize("T,D", [(1, 1), (1, 7), (7, 1), (5, 9), (64, 64), (100, 37), (37, 100), (300, 1000), (1024, 1024)])
def test_continuous_scores_equal_oracle(T, D, mask_kind, q):
    """continuous random scores: the optimum is unique almost surely, so the indices must be the oracle's"""
    rng = np.random.default_rng(T * 7919 + D * 31 + q + len(mask_kind))
    S = rng.normal(size=(T, D)).astype(np.float32)
    _check_equal_to_oracle(S, _mask(mask_kind, T, D, rng), q)


def test_full_size_equals_oracle():
    rng = np.random.default_rng(4096)
    S = rng.normal(size=(4096, 4096)).astype(np.float32)
    _check_equal_to_oracle(S, _mask("class8", 4096, 4096, rng), 10)


@pytest.mark.parametrize("mask_kind", ["none", "half", "class8"])
@pytest.mark.parametrize("T,D", [(6, 6), (40, 25), (25, 40), (200, 200), (512, 300)])
def test_integer_scores_ties_objective_exact_and_deterministic(T, D, mask_kind):
    """scores in [-3, 3]: many optimal matchings; any may come back, but it is valid, its objective is exactly the oracle's
    and two launches return the same bits"""
    rng = np.random.default_rng(T + 1000 * D + len(mask_kind))
    S = rng.integers(-3, 4, size=(T, D)).astype(np.float32)
    mask = _mask(mask_kind, T, D, rng)
    for tau in (-1.0, 0.0):
        d4t, t4d = _solve(S, tau, mask)
        assert R.consistent(d4t, t4d)
        rd, _ = R.assign(S, tau, mask)
        assert R.objective(S, tau, d4t, mask) == R.objective(S, tau, rd, mask)
        d2, t2 = _solve(S, tau, mask)
        assert np.array_equal(d4t, d2) and np.array_equal(t4d, t2)


def test_degenerate_inputs():
    from pcreid_b200.kernels import linear_assignment
    for T, D in ((0, 0), (0, 5), (5, 0)):
        d4t, t4d = linear_assignment(torch.zeros((T, D), device=DEV), 0.0)
        assert d4t.shape == (T,) and t4d.shape == (D,)
        assert (d4t == -1).all() and (t4d == -1).all()
        d4t, t4d = linear_assignment(torch.zeros((3, T, D), device=DEV), 0.0)
        assert d4t.shape == (3, T) and t4d.shape == (3, D)
    # everything inadmissible: below or at the threshold, masked out, non-finite
    S = np.full((4, 6), -1.0, np.float32)
    d4t, t4d = _solve(S, -1.0)
    assert (d4t == -1).all() and (t4d == -1).all()
    d4t, _ = _solve(np.ones((4, 6), np.float32), 0.0, np.zeros((4, 6), bool))
    assert (d4t == -1).all()
    d4t, _ = _solve(np.array([[np.nan, np.inf], [-np.inf, np.nan]], np.float32), 0.0)
    assert (d4t == -1).all()
    # all scores equal: a maximum matching
    for T, D in ((5, 5), (3, 8), (8, 3), (100, 100)):
        d4t, t4d = _solve(np.full((T, D), 2.0, np.float32), 0.5)
        assert R.consistent(d4t, t4d) and (d4t >= 0).sum() == min(T, D)
    # NaN / inf entries among continuous scores: never matched, the rest equals the oracle
    rng = np.random.default_rng(9)
    S = rng.normal(size=(50, 60)).astype(np.float32)
    S.flat[rng.choice(S.size, 300, replace=False)] = rng.choice([np.nan, np.inf, -np.inf], 300)
    d4t, t4d = _solve(S, -0.5)
    rd, rt = R.assign(S, -0.5)
    assert np.array_equal(d4t, rd) and np.array_equal(t4d, rt)
    assert all(np.isfinite(S[t, d]) for t, d in enumerate(d4t) if d >= 0)


def test_batch_independence():
    """37 different problems in one launch == each problem solved alone (ties included)"""
    from pcreid_b200.kernels import linear_assignment
    rng = np.random.default_rng(37)
    S = rng.integers(-3, 4, size=(37, 50, 60)).astype(np.float32)
    S[::2] = rng.normal(size=(19, 50, 60)).astype(np.float32)
    lt, ld = rng.integers(0, 8, (37, 50)), rng.integers(0, 8, (37, 60))
    mask = torch.from_numpy(lt[:, :, None] == ld[:, None, :]).to(DEV)
    Sd = torch.from_numpy(S).to(DEV)
    d4t, t4d = linear_assignment(Sd, -0.5, mask)
    assert d4t.shape == (37, 50) and t4d.shape == (37, 60)
    for b in range(37):
        db, tb = linear_assignment(Sd[b], -0.5, mask[b])
        assert torch.equal(db, d4t[b]) and torch.equal(tb, t4d[b])
        if b % 2 == 0:
            rd, rt = R.assign(S[b], -0.5, mask[b].cpu().numpy())
            assert np.array_equal(db.cpu().numpy(), rd)


def test_no_host_synchronisation_and_graph_capture():
    from pcreid_b200.kernels import linear_assignment
    rng = np.random.default_rng(5)
    S = torch.from_numpy(rng.normal(size=(4, 96, 80)).astype(np.float32)).to(DEV)
    mask = torch.from_numpy(rng.random((4, 96, 80)) < 0.6).to(DEV)
    ref = linear_assignment(S, 0.1, mask)                       # warm-up: loads the library and the kernel
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = linear_assignment(S, 0.1, mask)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        linear_assignment(S, 0.1, mask)
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = linear_assignment(S, 0.1, mask)
    S.copy_(torch.flip(S, (0,)))
    mask.copy_(torch.flip(mask, (0,)))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out[0], torch.flip(ref[0], (0,))) and torch.equal(out[1], torch.flip(ref[1], (0,)))


def test_opcheck_lsap():
    from pcreid_b200 import _lib
    rng = np.random.default_rng(6)
    B, T, D = 2, 9, 7
    S = torch.from_numpy(rng.normal(size=(B, T, D)).astype(np.float32)).to(DEV)
    mask = torch.from_numpy(rng.random((B, T, D)) < 0.7).to(DEV)
    work = torch.empty(B * _lib.lib().pcreid_lsap_workspace_bytes(T, D), dtype=torch.uint8, device=DEV)
    d4t = torch.empty((B, T), dtype=torch.int32, device=DEV)
    t4d = torch.empty((B, D), dtype=torch.int32, device=DEV)
    torch.library.opcheck(torch.ops.pcreid.lsap.default, (B, T, D, S, mask, -0.2, d4t, t4d, work),
                          test_utils=("test_schema", "test_faketensor", "test_autograd_registration", "test_aot_dispatch_dynamic"))
    torch.ops.pcreid.lsap(B, T, D, S, mask, -0.2, d4t, t4d, work)
    for b in range(B):
        rd, rt = R.assign(S[b].cpu().numpy(), -0.2, mask[b].cpu().numpy())
        assert np.array_equal(d4t[b].cpu().numpy(), rd) and np.array_equal(t4d[b].cpu().numpy(), rt)


def test_argument_checks():
    from pcreid_b200.kernels import linear_assignment
    S = torch.zeros((3, 4), device=DEV)
    with pytest.raises(TypeError):
        linear_assignment(S.double(), 0.0)
    with pytest.raises(RuntimeError):
        linear_assignment(S.cpu(), 0.0)
    with pytest.raises(ValueError):
        linear_assignment(S[0], 0.0)
    with pytest.raises(ValueError):
        linear_assignment(S, float("nan"))
    with pytest.raises(TypeError):
        linear_assignment(S, torch.tensor(0.0, device=DEV))
    with pytest.raises(ValueError):
        linear_assignment(S, 0.0, torch.ones((4, 3), dtype=torch.bool, device=DEV))
    with pytest.raises(ValueError):
        linear_assignment(S, 0.0, torch.ones((3, 4), dtype=torch.uint8, device=DEV))
    with pytest.raises(ValueError):
        linear_assignment(torch.zeros((4097, 1), device=DEV), 0.0)


def test_match_all_pairs_with_class_gate_then_assignment():
    """end to end in parity_tc: gated logits of synthetic objects -> assignment == the oracle's on that very cost matrix"""
    from pcreid_b200.kernels import linear_assignment
    from pcreid_b200.models.tracking import class_gate
    m, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    m.set_mode("parity_tc")
    t, d = O.synth_objects(24, 128, 20), O.synth_objects(30, 128, 21)
    xt, ht = m.encode(t.to(DEV))
    xd, hd = m.encode(d.to(DEV))
    g = torch.Generator().manual_seed(2)
    tl, dl = torch.randint(0, 3, (24,), generator=g).to(DEV), torch.randint(0, 3, (30,), generator=g).to(DEV)
    gate = class_gate(dl, tl, torch.full((30,), 128, device=DEV), torch.full((24,), 128, device=DEV))
    cost = m.match_all_pairs(ht, xt, hd, xd, pair_mask=gate)
    c = cost.cpu().numpy()
    tau = float(np.float32(np.median(c[gate.cpu().numpy()])))
    d4t, t4d = linear_assignment(cost, tau, gate)
    rd, rt = R.assign(c, tau, gate.cpu().numpy())
    assert np.array_equal(d4t.cpu().numpy(), rd) and np.array_equal(t4d.cpu().numpy(), rt)
    assert (rd >= 0).any()


def test_step_over_two_frames_equals_manual_composition():
    from test_frontend_oracle import scene
    from pcreid_b200.models.tracking import PointFeatureSet, PointReidentifier, class_gate
    m, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    bank = PointFeatureSet()
    xt, ht = m.encode(O.synth_objects(6, 128, 40).to(DEV))
    bank.store_new(xt, ht, torch.tensor([128, 20, 128, 5, 128, 60], device=DEV))
    manual = copy.deepcopy(bank)
    reid = PointReidentifier(m, bank, subsample_number=128)
    ref = PointReidentifier(m, manual, subsample_number=128)
    track_index = torch.tensor([0, 1, 2, 3, 4, 5], device=DEV)
    track_labels = torch.tensor([0, 1, 2, 0, 1, 2], device=DEV)
    for frame in range(2):
        pts, boxes = scene(60000, 9, 50 + frame)
        bt, pt = torch.from_numpy(boxes).to(DEV), torch.from_numpy(pts).to(DEV)
        rank = torch.randint(0, 1 << 30, (9, 128), generator=torch.Generator().manual_seed(frame))
        dl = torch.tensor([0, 1, 2, 0, 1, 2, 0, 1, 9], device=DEV)
        track_for_det, new_rows, cost = reid.step(pt, bt, dl, track_index, track_labels, -2.0, sample_rank=rank)
        # by hand: from_sweep + oracle + the bank's own methods on the copy
        cost2, xyz_d, h_d, len_d = ref.from_sweep(pt, bt, dl, track_index, track_labels, sample_rank=rank)
        assert torch.equal(cost, cost2)
        gate = class_gate(dl, track_labels, len_d, manual.lengths[track_index])
        _, rt = R.assign(cost2.cpu().numpy(), np.float32(-2.0), gate.cpu().numpy())
        assert track_for_det.cpu().tolist() == rt.tolist()
        rt = torch.from_numpy(rt).to(DEV)
        mt, un = torch.nonzero(rt >= 0).squeeze(1), torch.nonzero(rt < 0).squeeze(1)
        manual.replace_old(track_index[rt[mt]], xyz_d[mt], h_d[mt], len_d[mt])
        first = len(manual)
        manual.store_new(xyz_d[un], h_d[un], len_d[un])
        assert new_rows.cpu().tolist() == list(range(first, first + un.numel()))
        assert torch.equal(bank.pts_xyz, manual.pts_xyz) and torch.equal(bank.pts_feats, manual.pts_feats)
        assert torch.equal(bank.lengths, manual.lengths)
        assert int(track_for_det[8]) == -1                                     # class 9 is never compared
        track_index = torch.cat([track_index, new_rows])
        track_labels = torch.cat([track_labels, dl[un]])
