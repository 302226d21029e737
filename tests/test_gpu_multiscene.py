"""-m gpu: many scenes in one tracker step.  The segmented crop front-end against per-sweep crop_center_resample, block-batched
assignment against linear_assignment per problem, match_pairs against match_all_pairs, and MultiScenePointReidentifier.step
against one PointReidentifier.step per scene -- all bit for bit -- plus the launch counts that must not grow with the scene
count."""
import copy

import numpy as np
import pytest
import torch

import helpers
from oracle import reid_oracle as O
from test_frontend_oracle import scene

pytestmark = pytest.mark.gpu
DEV = "cuda"


# ---------------------------------------------------------------------------------------------------------- fixtures
def _scenes(sizes, seed):
    """[(pts (P, 4), boxes (B, 7))] on the device; some boxes are moved far away so that they hold no point"""
    out = []
    for k, (P, B) in enumerate(sizes):
        pts, boxes = scene(P, B, seed + k)
        if B > 1:
            boxes[::3, :2] += 500.0
        out.append((torch.from_numpy(pts).to(DEV), torch.from_numpy(boxes).to(DEV)))
    return out


def _ranks(B, N, seed):
    return torch.randint(0, 1 << 30, (B, N), generator=torch.Generator().manual_seed(seed)).to(DEV)


@pytest.fixture(scope="module")
def pt_model():
    m, _ = helpers.build_pair("pt", (128, 64, 32), device=DEV)
    return m


# ---------------------------------------------------------------------------------------------------------- front-end
SWEEPS = [0, 1, 1023, 1024, 1025, 60000]


@pytest.mark.parametrize("S", [1, 2, 6, 17, 33])
def test_segmented_crop_equals_per_sweep(S):
    from pcreid_b200 import _lib
    from pcreid_b200.models.frontend import _OPS, crop_center_resample, crop_center_resample_scenes, points_in_boxes_mask
    rng = np.random.default_rng(S)
    sizes = [(SWEEPS[(S + k) % len(SWEEPS)] if k % 5 else int(rng.integers(0, 3000)), int(rng.integers(0, 40)) if k % 4 else 0)
             for k in range(S)]
    sizes[0] = (60000, 37)                      # a full sweep with 37 boxes in every launch: some boxes hold points
    sc = _scenes(sizes, 100 * S)
    N = 64
    ranks = [_ranks(B, N, 7 * S + k) for k, (_, B) in enumerate(sizes)]
    pts = torch.cat([p for p, _ in sc])
    boxes = torch.cat([b for _, b in sc])
    out, lengths = crop_center_resample_scenes(boxes, pts, [B for _, B in sizes], [P for P, _ in sizes], N,
                                               sample_rank=torch.cat(ranks))
    # mask words and counts of the segmented pass: each box's block equals pcreid_crop_mask's on its own sweep
    L = _lib.lib()
    nt = [L.pcreid_crop_tiles(P) for P, _ in sizes]
    offs = [[0] for _ in range(4)]
    for (P, B), t in zip(sizes, nt):
        for row, v in zip(offs, (P, B, t, B * t)):
            row.append(row[-1] + v)
    C = offs[3][-1]
    mask = torch.full((C, 32), -7, device=DEV, dtype=torch.int32)
    counts = torch.full((C,), -7, device=DEV, dtype=torch.int32)
    _OPS.crop_mask_scenes(S, offs[2][-1], max(B for _, B in sizes), pts, pts.shape[1], boxes,
                          torch.tensor(offs, dtype=torch.int32, device=DEV), mask, counts)
    g0 = 0
    for k, ((p, b), (P, B)) in enumerate(zip(sc, sizes)):
        o1, l1 = crop_center_resample(b, p, N, sample_rank=ranks[k])
        assert torch.equal(out[g0:g0 + B], o1[0]) and torch.equal(lengths[g0:g0 + B], l1[0]), (k, P, B)
        if P and B:
            m1, c1, _ = points_in_boxes_mask(b, p)
            c0 = offs[3][k]
            assert torch.equal(mask[c0:c0 + B * nt[k]].view(B, nt[k], 32), m1)
            assert torch.equal(counts[c0:c0 + B * nt[k]].view(B, nt[k]), c1)
        g0 += B
    assert (lengths == 0).any() and (lengths > 0).any()


def test_segmented_crop_drawn_ranks_are_in_range():
    from pcreid_b200.models.frontend import crop_center_resample, crop_center_resample_scenes
    sc = _scenes([(5000, 6), (0, 3), (3000, 5)], 9)
    out, lengths = crop_center_resample_scenes(torch.cat([b for _, b in sc]), torch.cat([p for p, _ in sc]), [6, 3, 5],
                                               [5000, 0, 3000], 32)
    g0 = 0
    for p, b in sc:
        B = b.shape[0]
        _, l1 = crop_center_resample(b, p, 32)
        assert torch.equal(lengths[g0:g0 + B], l1[0])
        assert torch.equal(out[g0:g0 + B][l1[0] == 0], torch.zeros_like(out[g0:g0 + B][l1[0] == 0]))
        g0 += B


# ---------------------------------------------------------------------------------------------------------- assignment
def _problems(shapes, kind, seed, masked):
    g = torch.Generator().manual_seed(seed)
    blocks, masks = [], []
    for T, D in shapes:
        s = torch.randn(T, D, generator=g) if kind == "cont" else torch.randint(-2, 3, (T, D), generator=g).float()
        blocks.append(s.to(DEV))
        masks.append((torch.rand(T, D, generator=g) < 0.6).to(DEV) if masked else None)
    return blocks, masks


def _packed(blocks, masks):
    score = torch.cat([b.reshape(-1) for b in blocks])
    mask = None if masks[0] is None else torch.cat([m.reshape(-1) for m in masks])
    return score, mask


RAGGED = [(0, 5), (5, 0), (1, 1), (0, 0), (3, 17), (17, 3), (64, 64), (200, 130), (31, 33), (1024, 700), (2, 900), (700, 2)]


@pytest.mark.parametrize("kind", ["cont", "int"])
@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("shapes", [RAGGED, [(4096, 4096), (3, 5), (0, 7), (40, 40)]], ids=["ragged", "large"])
def test_lsap_blocks_equals_per_problem(kind, masked, shapes):
    from pcreid_b200.kernels import linear_assignment, linear_assignment_blocks
    blocks, masks = _problems(shapes, kind, len(shapes) + masked, masked)
    score, mask = _packed(blocks, masks)
    tau = -0.5 if kind == "cont" else 0.0
    d4t, t4d = linear_assignment_blocks(score, shapes, tau, mask)
    assert d4t.dtype == torch.int64 and d4t.shape == (sum(t for t, _ in shapes),) and t4d.shape == (sum(d for _, d in shapes),)
    r0 = c0 = 0
    for (T, D), s, m in zip(shapes, blocks, masks):
        rd, rt = linear_assignment(s, tau, m)
        assert torch.equal(d4t[r0:r0 + T], rd) and torch.equal(t4d[c0:c0 + D], rt), (T, D)
        r0, c0 = r0 + T, c0 + D
    # bit-identical relaunch
    d2, t2 = linear_assignment_blocks(score, shapes, tau, mask)
    assert torch.equal(d2, d4t) and torch.equal(t2, t4d)


def test_lsap_blocks_result_independent_of_neighbours():
    """problem (200, 130) alone, beside small problems, and beside a 4096-column problem (other thread count, shared memory)"""
    from pcreid_b200.kernels import linear_assignment_blocks
    (s,), (m,) = _problems([(200, 130)], "int", 5, True)
    ref = None
    for before, after in (([], []), ([(3, 4)], [(1, 1)]), ([(10, 4096)], [(0, 3), (50, 60)])):
        bb, mb = _problems(before, "int", 6, True) if before else ([], [])
        ba, ma = _problems(after, "int", 7, True) if after else ([], [])
        score, mask = _packed(bb + [s] + ba, mb + [m] + ma)
        d4t, t4d = linear_assignment_blocks(score, before + [(200, 130)] + after, 0.0, mask)
        r0, c0 = sum(t for t, _ in before), sum(d for _, d in before)
        got = (d4t[r0:r0 + 200], t4d[c0:c0 + 130])
        if ref is None:
            ref = got
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])


def test_lsap_blocks_no_host_synchronisation_and_opcheck():
    from pcreid_b200 import _lib
    from pcreid_b200.kernels import linear_assignment_blocks
    shapes = [(3, 5), (0, 4), (6, 6), (2, 0)]
    blocks, masks = _problems(shapes, "cont", 11, True)
    score, mask = _packed(blocks, masks)
    linear_assignment_blocks(score, shapes, 0.0, mask)                     # warm-up: library load, pinned buffers
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        d4t, t4d = linear_assignment_blocks(score, shapes, 0.0, mask)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert d4t.shape == (11,) and t4d.shape == (15,)
    L = _lib.lib()
    offs = [[0] for _ in range(4)]
    for T, D in shapes:
        for row, v in zip(offs, (T, D, T * D, L.pcreid_lsap_workspace_bytes(T, D))):
            row.append(row[-1] + v)
    args = (len(shapes), 6, 6, torch.tensor(offs, dtype=torch.int64, device=DEV), score, mask, 0.0,
            torch.empty(11, dtype=torch.int32, device=DEV), torch.empty(15, dtype=torch.int32, device=DEV),
            torch.empty(offs[3][-1], dtype=torch.uint8, device=DEV))
    torch.library.opcheck(torch.ops.pcreid.lsap_blocks, args, test_utils=("test_schema", "test_faketensor"))


def test_lsap_blocks_argument_checks():
    from pcreid_b200.kernels import linear_assignment_blocks
    s = torch.zeros(6, device=DEV)
    with pytest.raises(ValueError):
        linear_assignment_blocks(s, [(2, 2)], 0.0)                          # 6 elements for 4
    with pytest.raises(ValueError):
        linear_assignment_blocks(s, [(2, 3)], float("nan"))
    with pytest.raises(ValueError):
        linear_assignment_blocks(torch.zeros(4097, device=DEV), [(4097, 1)], 0.0)
    with pytest.raises(ValueError):
        linear_assignment_blocks(s, [(2, 3)], 0.0, torch.ones(6, device=DEV))   # mask not bool
    with pytest.raises(TypeError):
        linear_assignment_blocks(s, [(2, 3)], torch.tensor(0.0))


# ---------------------------------------------------------------------------------------------------------- match_pairs
@pytest.mark.parametrize("mode", ["parity", "parity_tc", "fast"])
def test_match_pairs_equals_match_all_pairs(pt_model, mode):
    from pcreid_b200.models.tracking import class_gate
    m = pt_model.set_mode(mode)
    xt, ht = m.encode(O.synth_objects(13, 128, 30).to(DEV))
    xd, hd = m.encode(O.synth_objects(11, 128, 31).to(DEV))
    g = torch.Generator().manual_seed(3)
    gate = class_gate(torch.randint(0, 3, (11,), generator=g).to(DEV), torch.randint(0, 3, (13,), generator=g).to(DEV),
                      None, None, use_lengths=False)
    dense = m.match_all_pairs(ht, xt, hd, xd, pair_mask=gate)
    nz = gate.nonzero()
    perm = torch.randperm(nz.shape[0], generator=g).to(DEV)
    nz = torch.cat([nz[perm], nz[:5]])                                      # unsorted, with repeats
    got = m.match_pairs(ht, xt, hd, xd, nz[:, 0], nz[:, 1])
    assert torch.equal(got, dense[nz[:, 0], nz[:, 1]])
    m.set_mode("parity")


# ---------------------------------------------------------------------------------------------------------- tracker step
def _run_steps(model, sizes, mode, replace_all, n_frames=3, min_score=-2.0, seed=0):
    """S scenes over n_frames: MultiScenePointReidentifier.step against one PointReidentifier.step per scene, bit for bit"""
    from pcreid_b200.models.tracking import MultiScenePointReidentifier, PointFeatureSet, PointReidentifier
    model.set_mode(mode)
    S = len(sizes)
    banks = []
    for s, (_, _, T) in enumerate(sizes):
        bank = PointFeatureSet(replace_all)
        if T:
            x, h = model.encode(O.synth_objects(T, 128, 500 + s).to(DEV))
            bank.store_new(x, h, 100 + torch.arange(T, device=DEV) % 7)
        banks.append(bank)
    ref_banks = copy.deepcopy(banks)
    multi = MultiScenePointReidentifier(model, banks)
    track_index = [torch.arange(T, device=DEV) for _, _, T in sizes]
    track_labels = [torch.arange(T, device=DEV) % 3 for _, _, T in sizes]
    matched = 0
    for frame in range(n_frames):
        sc = _scenes([(P, B) for P, B, _ in sizes], seed + 1000 * frame)
        frames, ranks = [], []
        for s, (pts, boxes) in enumerate(sc):
            B = boxes.shape[0]
            dl = torch.arange(B, device=DEV) % 3
            if B:
                dl[-1] = 9                                                  # never compared
            none = S > 2 and s == 2 and frame == 1                          # a scene with nothing this step
            frames.append(None if none else (pts, boxes, dl, track_index[s], track_labels[s]))
            ranks.append(None if none else _ranks(B, 128, 31 * s + frame))
        got = multi.step(frames, min_score, sample_ranks=ranks)
        for s in range(S):
            if frames[s] is None:
                assert got[s] is None
                continue
            want = PointReidentifier(model, ref_banks[s]).step(*frames[s], min_score, sample_rank=ranks[s])
            for a, b in zip(got[s], want):
                assert (a is None) == (b is None), (frame, s)
                if a is not None:
                    assert torch.equal(a, b), (mode, frame, s)
            bank, rb = banks[s], ref_banks[s]
            assert len(bank) == len(rb)
            if len(rb):
                assert torch.equal(bank.pts_xyz, rb.pts_xyz) and torch.equal(bank.pts_feats, rb.pts_feats)
                assert torch.equal(bank.lengths, rb.lengths)
            tfd = got[s][0]
            if tfd.numel():
                assert int(tfd[-1]) == -1
            matched += int((tfd >= 0).sum())
            un = torch.nonzero(tfd < 0).squeeze(1)
            track_index[s] = torch.cat([track_index[s], got[s][1]])
            track_labels[s] = torch.cat([track_labels[s], frames[s][2][un]])
    model.set_mode("parity")
    return matched


# (points, boxes, tracks at the start) per scene: scene 1 has no tracks, scene 3 no detections, scene 2 is None in frame 1
SIZES = [(20000, 9, 6), (5000, 7, 0), (60000, 12, 8), (3000, 0, 4), (1025, 5, 3)]


@pytest.mark.parametrize("mode", ["parity", "parity_tc", "fast"])
@pytest.mark.parametrize("replace_all", [False, True])
def test_multiscene_step_equals_per_scene_steps(pt_model, mode, replace_all):
    assert _run_steps(pt_model, SIZES, mode, replace_all) > 0


def test_multiscene_step_one_scene(pt_model):
    _run_steps(pt_model, SIZES[:1], "parity_tc", False)


def test_multiscene_step_17_scenes(pt_model):
    rng = np.random.default_rng(17)
    sizes = [(int(rng.integers(0, 30000)), int(rng.integers(0, 14)), int(rng.integers(0, 10))) for _ in range(17)]
    assert _run_steps(pt_model, sizes, "parity_tc", False, seed=17) > 0


def test_multiscene_step_concat_model():
    m, _ = helpers.build_pair("concat", (128, 64, 32), device=DEV)
    for mode in ("parity", "fast"):
        _run_steps(m, SIZES, mode, False)


def test_launches_do_not_grow_with_scene_count(pt_model, monkeypatch):
    """crop mask, crop gather and lsap run once per step for 1 and for 17 scenes; the fused matcher's launches do not grow"""
    from pcreid_b200 import torch_ops
    from pcreid_b200.models import frontend
    import pcreid_b200.kernels as K
    counted = ("crop_mask_scenes", "crop_gather_scenes", "lsap_blocks", "pair_p1a2", "pair_p1b_n", "pair_p2y", "crop_mask",
               "crop_gather", "lsap")
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

    monkeypatch.setattr(frontend, "_OPS", Counting())
    monkeypatch.setattr(K, "_OPS", Counting())
    from pcreid_b200.models import fused_pairs
    if hasattr(fused_pairs, "_OPS"):
        monkeypatch.setattr(fused_pairs, "_OPS", Counting())
    per_S = {}
    for S in (1, 17):
        rng = np.random.default_rng(S)
        sizes = [(int(rng.integers(1000, 20000)), int(rng.integers(2, 10)), int(rng.integers(2, 8))) for _ in range(S)]
        _run_steps(pt_model, sizes, "parity_tc", False, n_frames=1)         # warm-up (per-scene steps count too)
        calls.clear()
        from pcreid_b200.models.tracking import MultiScenePointReidentifier, PointFeatureSet
        pt_model.set_mode("parity_tc")
        banks = []
        for s, (_, _, T) in enumerate(sizes):
            bank = PointFeatureSet()
            x, h = pt_model.encode(O.synth_objects(T, 128, 900 + s).to(DEV))
            bank.store_new(x, h, torch.full((T,), 128, device=DEV))
            banks.append(bank)
        sc = _scenes([(P, B) for P, B, _ in sizes], 77)
        frames = [(p, b, torch.arange(b.shape[0], device=DEV) % 3, torch.arange(T, device=DEV), torch.arange(T, device=DEV) % 3)
                  for (p, b), (_, _, T) in zip(sc, sizes)]
        calls.clear()
        MultiScenePointReidentifier(pt_model, banks).step(frames, -2.0)
        pt_model.set_mode("parity")
        per_S[S] = dict(calls)
    for S in (1, 17):
        assert per_S[S].get("crop_mask_scenes") == 1 and per_S[S].get("crop_gather_scenes") == 1, per_S
        assert per_S[S].get("lsap_blocks") == 1 and "lsap" not in per_S[S] and "crop_mask" not in per_S[S], per_S
    fused = ("pair_p1a2", "pair_p1b_n", "pair_p2y")
    assert sum(per_S[1].get(k, 0) for k in fused) > 0
    assert all(per_S[17].get(k, 0) == per_S[1].get(k, 0) for k in fused), per_S
