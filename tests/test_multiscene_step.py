"""CPU checks of the multi-scene tracker step (models/tracking.py, MultiScenePointReidentifier): the segmented front-end, the
encoder and the pair scorer are replaced by fixed tensors, kernels.linear_assignment(_blocks) by the scipy oracle
(tests/assign_reference.py, tests/assign_blocks_reference.py).  Every scene's outputs and bank must equal those of its own PointReidentifier.step.  Also the
argument handling of the new C entry points (pcreid_lsap_blocks, pcreid_crop_*_scenes), answered before any CUDA call."""
import copy

import numpy as np
import pytest
import torch

import assign_blocks_reference as RB
import assign_reference as R

N = 16


def _logits(h_t, h_d, ti, dj):
    """the fake pair scorer: one fixed function of the two objects' features (elementwise: no reduction whose order could
    depend on the number of pairs)"""
    return h_t[ti, 0, 0] * h_d[dj, 0, 0] + h_t[ti, 1, 1] - h_d[dj, 2, 3]


class FakeModel:
    match_type = "xcorr_eff"

    def encode(self, pts):
        return pts, pts.permute(0, 2, 1) * 0.5

    def match_pairs(self, h_t, xyz_t, h_d, xyz_d, ti, dj, chunk=8192):
        return _logits(h_t, h_d, ti, dj)

    def match_all_pairs(self, h_t, xyz_t, h_d, xyz_d, pair_mask=None):
        out = torch.zeros((h_t.shape[0], h_d.shape[0]))
        nz = pair_mask.nonzero()
        out[nz[:, 0], nz[:, 1]] = _logits(h_t, h_d, nz[:, 0], nz[:, 1])
        return out


def _scene(s, frame, D, T_bank):
    """fixed detections of scene s: (points (D, N, 3), lengths (D,), labels (D,))"""
    g = torch.Generator().manual_seed(1000 * s + frame)
    pts = torch.randn(D, N, 3, generator=g)
    lengths = torch.randint(0, 6, (D,), generator=g)
    labels = torch.randint(0, 3, (D,), generator=g)
    if D:
        labels[-1] = 9                                                  # never compared
    return pts, lengths, labels


def _bank(s, T, replace_all):
    from pcreid_b200.models.tracking import PointFeatureSet
    bank = PointFeatureSet(replace_all)
    if T:
        g = torch.Generator().manual_seed(77 + s)
        x = torch.randn(T, N, 3, generator=g)
        bank.store_new(x, x.permute(0, 2, 1) * 0.5, torch.randint(0, 6, (T,), generator=g))
    return bank


@pytest.mark.parametrize("replace_all", [False, True])
@pytest.mark.parametrize("min_score", [0.5, -2.0])
def test_multiscene_step_equals_per_scene_steps(monkeypatch, replace_all, min_score):
    import pcreid_b200.kernels as K
    import pcreid_b200.models.tracking as TR
    monkeypatch.setattr(K, "linear_assignment", R.linear_assignment)
    monkeypatch.setattr(K, "linear_assignment_blocks", RB.linear_assignment_blocks)
    # per scene: detections per frame, tracks in the bank at the start; scene 2 has no tracks, scene 3 no detections,
    # scene 4 is None in frame 1
    dets = [5, 3, 4, 0, 6, 1]
    tracks = [4, 2, 0, 3, 5, 1]
    S = len(dets)
    model = FakeModel()
    banks = [_bank(s, tracks[s], replace_all) for s in range(S)]
    ref_banks = copy.deepcopy(banks)
    multi = TR.MultiScenePointReidentifier(model, banks)
    track_index = [torch.arange(tracks[s]) for s in range(S)]
    track_labels = [torch.arange(tracks[s]) % 3 for s in range(S)]
    for frame in range(3):
        data = [_scene(s, frame, dets[s], tracks[s]) for s in range(S)]
        frames = [None if (s == 4 and frame == 1) else
                  (torch.zeros(0, 4), torch.zeros(dets[s], 7), data[s][2], track_index[s], track_labels[s]) for s in range(S)]
        # the fake front-end returns each scene's fixed points and lengths, concatenated in scene order
        live = [s for s in range(S) if frames[s] is not None]
        monkeypatch.setattr(TR, "crop_center_resample_scenes", lambda *a, **kw: (
            torch.cat([data[s][0] for s in live]), torch.cat([data[s][1] for s in live])))
        got = multi.step(frames, min_score)
        for s in range(S):
            if frames[s] is None:
                assert got[s] is None
                continue
            ref = TR.PointReidentifier(model, ref_banks[s])

            def from_sweep(sweep, bboxes, det_labels, ti, tl, sample_rank=None, ref=ref, s=s):
                xyz_d, h_d = model.encode(data[s][0])
                if ti is None or len(ti) == 0:
                    return None, xyz_d, h_d, data[s][1]
                cost, _, _ = ref(data[s][0], det_labels, data[s][1], ti, tl)
                return cost, xyz_d, h_d, data[s][1]

            monkeypatch.setattr(ref, "from_sweep", from_sweep)
            want = ref.step(*frames[s], min_score)
            for a, b in zip(got[s], want):
                assert (a is None) == (b is None)
                if a is not None:
                    assert torch.equal(a, b), (frame, s)
            bank, rb = banks[s], ref_banks[s]
            assert len(bank) == len(rb)
            if len(rb):
                assert torch.equal(bank.pts_xyz, rb.pts_xyz) and torch.equal(bank.pts_feats, rb.pts_feats)
                assert torch.equal(bank.lengths, rb.lengths)
            if dets[s]:
                assert int(got[s][0][-1]) == -1                          # class 9
            # the unmatched detections become tracks of the next frame
            un = torch.nonzero(got[s][0] < 0).squeeze(1)
            track_index[s] = torch.cat([track_index[s], got[s][1]])
            track_labels[s] = torch.cat([track_labels[s], data[s][2][un]])
            tracks[s] = len(track_index[s])
    assert any(int((r[0] >= 0).sum()) for r in got if r is not None)        # some detections were matched


def test_multiscene_step_all_scenes_none():
    from pcreid_b200.models.tracking import MultiScenePointReidentifier, PointFeatureSet
    multi = MultiScenePointReidentifier(FakeModel(), [PointFeatureSet(), PointFeatureSet()])
    assert multi.step([None, None], 0.0) == [None, None]
    with pytest.raises(ValueError):
        multi.step([None], 0.0)


def test_blocks_stand_in_equals_per_problem_oracle():
    rng = np.random.default_rng(3)
    shapes = [(0, 3), (3, 0), (1, 1), (5, 7), (7, 5), (0, 0), (4, 4)]
    blocks = [rng.integers(-3, 4, (T, D)).astype(np.float32) for T, D in shapes]
    masks = [rng.random((T, D)) < 0.7 for T, D in shapes]
    score = torch.from_numpy(np.concatenate([b.reshape(-1) for b in blocks]))
    mask = torch.from_numpy(np.concatenate([m.reshape(-1) for m in masks]))
    d4t, t4d = RB.linear_assignment_blocks(score, shapes, -1.0, mask)
    assert d4t.dtype == torch.int64 and d4t.shape == (sum(t for t, _ in shapes),)
    assert t4d.shape == (sum(d for _, d in shapes),)
    r0 = c0 = 0
    for (T, D), b, m in zip(shapes, blocks, masks):
        rd, rt = R.assign(b, np.float32(-1.0), m)
        assert d4t[r0:r0 + T].tolist() == rd.tolist() and t4d[c0:c0 + D].tolist() == rt.tolist()
        r0, c0 = r0 + T, c0 + D


@pytest.fixture(scope="module")
def L():
    from pcreid_b200 import _lib
    return _lib.lib()


def test_lsap_blocks_argument_errors_before_any_cuda_call(L):
    f = L.pcreid_lsap_blocks
    args = lambda B, mt, md, tau=0.0: (B, mt, md, None, None, None, tau, None, None, None, None)
    # negative sizes, a non-finite threshold: PCREID_ERR_ARG
    for a in (args(-1, 4, 4), args(1, -4, 4), args(1, 4, -4), args(1, 4, 4, float("nan")), args(1, 4, 4, float("inf"))):
        assert f(*a) == 1
    # beyond the kernel: PCREID_ERR_UNSUPPORTED
    for a in (args(1, 4097, 4), args(1, 4, 4097), args(65536, 4, 4)):
        assert f(*a) == 3
    # null offsets / buffers: PCREID_ERR_ARG
    assert f(*args(1, 4, 4)) == 1
    assert f(*args(1, 0, 4)) == 1                        # track_for_det needed
    assert f(*args(1, 4, 0)) == 1                        # det_for_track and work needed
    # nothing to do: PCREID_OK without touching a pointer
    assert f(*args(0, 4, 4)) == 0
    assert f(*args(3, 0, 0)) == 0


def test_crop_scenes_argument_errors_before_any_cuda_call(L):
    m, g = L.pcreid_crop_mask_scenes, L.pcreid_crop_gather_scenes
    assert m(-1, 1, 1, None, 3, None, None, None, None, None) == 1
    assert m(1, -1, 1, None, 3, None, None, None, None, None) == 1
    assert m(1, 1, -1, None, 3, None, None, None, None, None) == 1
    assert m(1, 1, 1, None, 3, None, None, None, None, None) == 1
    assert m(1, 1, 65535 * 32 + 1, 1, 3, 1, 1, 1, 1, None) == 3
    assert m(0, 1, 1, None, 3, None, None, None, None, None) == 0
    assert m(2, 0, 5, None, 3, None, None, None, None, None) == 0       # empty sweeps: nothing to test
    assert g(-1, 1, 1, None, 3, None, None, None, None, None, None, None) == 1
    assert g(1, 1, -1, None, 3, None, None, None, None, None, None, None) == 1
    assert g(1, 1, 1, None, 3, None, None, None, None, None, None, None) == 1
    assert g(1, 65536, 1, 1, 3, 1, 1, 1, 1, 1, 1, None) == 3
    assert g(1, 0, 4, None, 3, None, None, None, None, None, None, None) == 0
