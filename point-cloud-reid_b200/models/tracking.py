"""The all-pairs driver pieces of the reference's deprecated tracker, on the accelerated path (SURVEY 8f rank 1):

* ``PointFeatureSet`` -- per-track bank of stage-0 embeddings (trackers/deprecated/tracking_feature_set.py:12-63):
  ``store_new`` appends, ``replace_old`` keeps the observation with more points (or always replaces).
* ``class_gate`` -- ``get_labels_to_compare`` (trackers/deprecated/tracking_point_reid.py:15-33) as a dense boolean (T, D)
  mask instead of a concatenated cartesian-product index list.
* ``PointReidentifier`` -- the scoring part of ``PointReidentifier.__call__`` (L88-116): encode the detections, gate,
  score every admissible track x detection pair, return the dense (T, D) cost matrix (zeros where not compared).
  ``from_sweep`` runs the whole of ``__call__`` (L74-116): crop / centre / resample the sweep with the fused front-end
  (models/frontend.py replaces pc_utils.py:31-96), then encode, gate and score.
  ``step`` is one tracker frame after that on the device: associate with ``kernels.linear_assignment`` (maximum-weight
  matching of the class-gated pairs whose logit exceeds ``min_score``), then update the bank as the reference's
  virtual_tracker.py:800-812 does -- matched detections through ``replace_old``, unmatched ones through ``store_new``.
  Track lifecycle (ids, ages, deletion, motion) stays with the caller.
* ``MultiScenePointReidentifier`` -- ``step`` over many independent scenes (one bank each) with one front-end pass, one
  encode, one pair-scoring call and one assignment launch for all of them; every scene's result and bank equal those of its
  own ``PointReidentifier.step``.
* ``score_pair_blocks`` -- the pair-list scorer both multi-scene classes share: one ``match_pairs`` call over the gated pairs
  of many packed (T_b, D_b) blocks.
* ``TrackTable`` / ``ReIDTracker`` -- the tracker that keeps its tracks: a device-resident table of S scenes x C slots (ids,
  labels, ages, hits, last boxes, bank rows) and a step that gates, scores, assigns and updates every scene with one launch
  of each kernel (kernels.track_gate_blocks / track_update / track_scatter) and no per-scene Python loop over tensors.
  Retirement after ``max_age`` unmatched steps, a bounded bank and an optional centre-distance gate come with it.
* ``MotionModel`` -- optional motion for ``ReIDTracker``: a constant-velocity Kalman filter per slot in the style of AB3DMOT,
  kept in the table (kernels.track_predict / track_correct).  Every active track is predicted before the gate, which then
  tests the predicted box (``max_distance``) and, optionally, the Mahalanobis distance of the predicted ground-plane centre.
"""
import math

import torch

from .. import kernels as K
from .frontend import crop_center_resample, crop_center_resample_scenes


class PointFeatureSet:
    def __init__(self, replace_all=False):
        self.replace_all = replace_all
        self.set_attributes()

    def set_attributes(self):
        self.pts_feats = None
        self.pts_xyz = None
        self.lengths = None

    def reset(self):
        self.set_attributes()

    def __len__(self):
        return 0 if self.pts_feats is None else self.pts_feats.shape[0]

    def get_features(self, index):
        return self.pts_xyz[index, ...], self.pts_feats[index, ...]

    def store_new(self, xyz, feats, lengths):
        if self.pts_feats is None:
            self.pts_feats, self.pts_xyz, self.lengths = feats, xyz, lengths
        else:
            self.pts_feats = torch.cat([self.pts_feats, feats], dim=0)
            self.pts_xyz = torch.cat([self.pts_xyz, xyz], dim=0)
            self.lengths = torch.cat([self.lengths, lengths], dim=0)

    def replace_old(self, index, xyz, feats, lengths):
        """Only replace the old features if the new observation has at least as many points (unless replace_all)."""
        if self.pts_feats is None:
            raise ValueError('pts_feats should not be None for replace_old')
        if not self.replace_all:
            keep = torch.where(self.lengths[index] <= lengths)[0]
            index, xyz, feats, lengths = index[keep], xyz[keep], feats[keep], lengths[keep]
        self.pts_feats[index, ...] = feats
        self.pts_xyz[index, ...] = xyz
        self.lengths[index, ...] = lengths


def class_gate(det_labels, track_labels, det_lengths=None, track_lengths=None, use_lengths=True, num_classes=8, min_points=2):
    """(T, D) bool: track t and detection d share a class in [0, num_classes) (and both have >= min_points points)."""
    ok_t = (track_labels >= 0) & (track_labels < num_classes)
    ok_d = (det_labels >= 0) & (det_labels < num_classes)
    if use_lengths:
        ok_t = ok_t & (track_lengths >= min_points)
        ok_d = ok_d & (det_lengths >= min_points)
    return (track_labels[:, None] == det_labels[None, :]) & ok_t[:, None] & ok_d[None, :]


def score_pair_blocks(model, gate, shapes, det_starts, h_t, xyz_t, h_d, xyz_d):
    """Logits of the gated pairs of many (T_b, D_b) blocks in one ``model.match_pairs`` call.  gate: bool, block b's row-major
    (T_b, D_b) mask after block b-1's (the packing of kernels.linear_assignment_blocks); block b's tracks are rows
    sum_{c<b} T_c .. of h_t / xyz_t, its detections rows det_starts[b] .. of h_d / xyz_d.
    -> packed float32 cost like gate: the logit where gate is set, 0 elsewhere."""
    dev = gate.device
    e_off, t_off = [0], [0]
    for T, D in shapes:
        e_off.append(e_off[-1] + T * D)
        t_off.append(t_off[-1] + T)
    meta = torch.tensor([e_off[:-1], t_off[:-1], list(det_starts), [D for _, D in shapes]], dtype=torch.int64).to(dev)
    e = gate.nonzero().squeeze(1)
    blk = torch.searchsorted(torch.tensor(e_off[1:], dtype=torch.int64).to(dev), e, right=True)
    local = e - meta[0, blk]
    ti = meta[1, blk] + local // meta[3, blk]
    dj = meta[2, blk] + local % meta[3, blk]
    cost = torch.zeros(gate.shape, device=dev, dtype=torch.float32)
    cost[e] = model.match_pairs(h_t, xyz_t, h_d, xyz_d, ti, dj)
    return cost


class PointReidentifier:
    """cost = reid(model, bank)(det_points, det_labels, det_lengths, track_index, track_labels)"""

    def __init__(self, model, feature_set=None, use_lengths=True, subsample_number=128):
        self.model = model
        self.feature_set = feature_set if feature_set is not None else PointFeatureSet(replace_all=False)
        self.use_lengths = use_lengths
        self.subsample_number = subsample_number

    @torch.no_grad()
    def from_sweep(self, sweep, bboxes, det_labels, track_index, track_labels, sample_rank=None):
        """sweep (P, >=3) LiDAR points, bboxes (D, 7) depth-frame boxes of the detections -> (cost (T, D) or None when
        there are no active tracks, xyz_det, feat_det, lengths_det): PointReidentifier.__call__
        (tracking_point_reid.py:74-116) from the raw sweep."""
        batch, lengths = crop_center_resample(bboxes[:, :7].float().contiguous(), sweep.float(), self.subsample_number,
                                              sample_rank=sample_rank)
        det_points, det_lengths = batch[0], lengths[0]
        if track_index is None or len(track_index) == 0:
            xyz_d, h_d = self.encode(det_points)
            return None, xyz_d, h_d, det_lengths
        cost, xyz_d, h_d = self(det_points, det_labels, det_lengths, track_index, track_labels)
        return cost, xyz_d, h_d, det_lengths

    @torch.no_grad()
    def step(self, sweep, bboxes, det_labels, track_index, track_labels, min_score, sample_rank=None):
        """One frame: from_sweep, association, bank update.  Track t (a position into ``track_index``) and detection d may be
        matched when the class gate allows it and cost[t, d] > min_score; the matching maximises the sum of
        cost - min_score.  Matched detections replace their track's bank row in one ``replace_old`` call (the bank's policy:
        the observation with more points is kept unless ``replace_all``); unmatched ones are appended with ``store_new``.
        -> (track_for_det (D,) int64 position into track_index or -1, new_rows (U,) int64 bank rows created for the
        unmatched detections in ascending detection order, cost (T, D) or None when there are no active tracks)."""
        cost, xyz_d, h_d, len_d = self.from_sweep(sweep, bboxes, det_labels, track_index, track_labels, sample_rank)
        dev = xyz_d.device
        if cost is None:
            track_for_det = torch.full((xyz_d.shape[0],), -1, dtype=torch.long, device=dev)
        else:
            # the gate matters: cost is 0 where a pair was not compared, and 0 can exceed a negative min_score
            gate = class_gate(det_labels, track_labels, len_d, self.feature_set.lengths[track_index], self.use_lengths)
            _, track_for_det = K.linear_assignment(cost, min_score, gate)
            matched = torch.nonzero(track_for_det >= 0).squeeze(1)
            self.feature_set.replace_old(track_index[track_for_det[matched]], xyz_d[matched], h_d[matched], len_d[matched])
        unmatched = torch.nonzero(track_for_det < 0).squeeze(1)
        first = len(self.feature_set)
        self.feature_set.store_new(xyz_d[unmatched], h_d[unmatched], len_d[unmatched])
        return track_for_det, torch.arange(first, first + unmatched.numel(), dtype=torch.long, device=dev), cost

    @torch.no_grad()
    def encode(self, det_points):
        return self.model.encode(det_points)

    @torch.no_grad()
    def __call__(self, det_points, det_labels, det_lengths, track_index, track_labels):
        """det_points (D, N, 3); track_index: rows of the feature bank of the active tracks.
        Returns (cost (T, D) with 0 where a pair is not compared, xyz_det, feat_det)."""
        xyz_d, h_d = self.encode(det_points)
        xyz_t, h_t = self.feature_set.get_features(track_index)
        mask = class_gate(det_labels, track_labels, det_lengths, self.feature_set.lengths[track_index], self.use_lengths)
        cost = self.model.match_all_pairs(h_t, xyz_t, h_d, xyz_d, pair_mask=mask)
        return cost, xyz_d, h_d


class MultiScenePointReidentifier:
    """PointReidentifier.step over S independent scenes at once: ``feature_sets[s]`` is scene s's bank (PointFeatureSet,
    unchanged semantics).  The crop front-end, the encoder, the pair scorer and the assignment each run once per step whatever
    S is (a 'concat' model scores scene by scene through its dense pooled head); the bank updates stay per scene."""

    def __init__(self, model, feature_sets, use_lengths=True, subsample_number=128):
        self.model = model
        self.feature_sets = list(feature_sets)
        self.use_lengths = use_lengths
        self.subsample_number = subsample_number

    @torch.no_grad()
    def step(self, frames, min_score, sample_ranks=None):
        """frames[s]: (sweep, bboxes, det_labels, track_index, track_labels) or None for a scene with nothing this step;
        sample_ranks: None (ranks drawn on the device) or one (D_s, N) int64 tensor per non-None scene.
        -> one (track_for_det, new_rows, cost) per scene, as PointReidentifier.step returns them (None for a None scene)."""
        if len(frames) != len(self.feature_sets):
            raise ValueError(f"{len(frames)} frames for {len(self.feature_sets)} scenes")
        live = [s for s, f in enumerate(frames) if f is not None]
        results = [None] * len(frames)
        if not live:
            return results
        if sample_ranks is not None and any(sample_ranks[s] is None for s in live):
            raise ValueError("sample_ranks must give ranks for every scene with a frame, or be None")
        sweeps = [frames[s][0].float() for s in live]
        boxes = [frames[s][1][:, :7].float() for s in live]
        n_det = [b.shape[0] for b in boxes]
        # 1. crop / centre / resample every scene's detections from its own sweep
        rank = None if sample_ranks is None else torch.cat([sample_ranks[s].to(sweeps[0].device, torch.int64) for s in live])
        det_points, det_len = crop_center_resample_scenes(torch.cat(boxes), torch.cat([w[:, :3] for w in sweeps]), n_det,
                                                          [w.shape[0] for w in sweeps], self.subsample_number, sample_rank=rank)
        # 2. one encode of all detections
        xyz_d, h_d = self.model.encode(det_points)
        d0 = [0]
        for n in n_det:
            d0.append(d0[-1] + n)
        # 3. the class gate of every scene with tracks, packed; their tracks from their own banks
        blocks, gates, xyz_t, h_t = [], [], [], []          # blocks: (scene, position in live, T_s, D_s)
        for k, s in enumerate(live):
            _, _, det_labels, track_index, track_labels = frames[s]
            if track_index is None or len(track_index) == 0:
                continue
            bank = self.feature_sets[s]
            xt, ht = bank.get_features(track_index)
            xyz_t.append(xt)
            h_t.append(ht)
            gates.append(class_gate(det_labels, track_labels, det_len[d0[k]:d0[k + 1]], bank.lengths[track_index],
                                    self.use_lengths))
            blocks.append((s, k, len(track_index), n_det[k]))
        costs = {}
        if blocks:
            cost, gate = self._score(blocks, gates, xyz_t, h_t, xyz_d, h_d, d0)
            # 6. one assignment launch over every scene's (T_s, D_s) problem
            _, tfd = K.linear_assignment_blocks(cost, [(T, D) for _, _, T, D in blocks], min_score, gate)
            e0 = c0 = 0
            for s, k, T, D in blocks:
                costs[s] = (cost[e0:e0 + T * D].view(T, D), tfd[c0:c0 + D])
                e0, c0 = e0 + T * D, c0 + D
        # 7. bank updates, per scene
        for k, s in enumerate(live):
            bank = self.feature_sets[s]
            sl = slice(d0[k], d0[k + 1])
            xd, hd, ld = xyz_d[sl], h_d[sl], det_len[sl]
            if s in costs:
                cost_s, track_for_det = costs[s]
                matched = torch.nonzero(track_for_det >= 0).squeeze(1)
                bank.replace_old(frames[s][3][track_for_det[matched]], xd[matched], hd[matched], ld[matched])
            else:
                cost_s = None
                track_for_det = torch.full((n_det[k],), -1, dtype=torch.long, device=xd.device)
            unmatched = torch.nonzero(track_for_det < 0).squeeze(1)
            first = len(bank)
            bank.store_new(xd[unmatched], hd[unmatched], ld[unmatched])
            results[s] = (track_for_det, torch.arange(first, first + unmatched.numel(), dtype=torch.long, device=xd.device),
                          cost_s)
        return results

    def _score(self, blocks, gates, xyz_t, h_t, xyz_d, h_d, d0):
        """-> (packed cost: each scene's row-major (T_s, D_s) logits, 0 where not compared; packed gate)"""
        gate = torch.cat([g.reshape(-1) for g in gates])
        if self.model.match_type == 'concat':
            # the dense pooled head scores whole blocks: scene by scene
            cost = torch.cat([self.model.match_all_pairs(ht, xt, h_d[d0[k]:d0[k + 1]], xyz_d[d0[k]:d0[k + 1]], pair_mask=g).reshape(-1)
                              for (_, k, _, _), g, xt, ht in zip(blocks, gates, xyz_t, h_t)])
            return cost, gate
        # 4. one match_pairs call over every scene's gated pairs; 5. logits scattered into the packed cost
        cost = score_pair_blocks(self.model, gate, [(T, D) for _, _, T, D in blocks], [d0[k] for _, k, _, _ in blocks],
                                 torch.cat(h_t), torch.cat(xyz_t), h_d, xyz_d)
        return cost, gate


class TrackTable:
    """Tracks of S scenes kept on the device: C slots per scene (1 <= C <= 4096), the state of kernels.TRACK_SLOT_FIELDS /
    TRACK_SCENE_FIELDS plus the bank rows ``xyz`` / ``feat`` (S * C rows; row r = s * C + slot), allocated from the first
    encode with its row shapes and dtypes.  A slot holds alive, track_id (unique within its scene, from 0, never reused),
    label, length (points of the kept observation), age (steps since the last match), hits and box (the last matched
    detection's 7 box values).  Per scene: next_id, dropped (detections that found no free slot), count and the active list
    ``active[s, :count[s]]`` (global rows of the alive slots, ascending).  Updated by ReIDTracker.step through
    kernels.track_update / track_scatter; the observation is replaced on a match when replace_all or when the new one has at
    least as many points (PointFeatureSet.replace_old's rule).

    With ``motion=True`` each slot also holds the state of kernels.TRACK_MOTION_FIELDS: the Kalman filter's box estimate
    ``kf_box``, velocity ``kf_vel`` and compact covariance ``kf_cov`` (include/pcreid.h), read with ``motion(s)``."""

    def __init__(self, num_scenes, capacity, replace_all=False, device="cuda", motion=False):
        if not 1 <= capacity <= K.TRACK_MAX_CAPACITY or not 1 <= num_scenes <= K.TRACK_MAX_SCENES:
            raise ValueError(f"TrackTable supports 1 <= capacity <= {K.TRACK_MAX_CAPACITY} and 1 <= num_scenes <= "
                             f"{K.TRACK_MAX_SCENES}; got {(num_scenes, capacity)}")
        self.num_scenes, self.capacity, self.replace_all = int(num_scenes), int(capacity), bool(replace_all)
        self.device = torch.device(device)
        self.has_motion = bool(motion)
        for name, dtype, tail in K.TRACK_SLOT_FIELDS + (K.TRACK_MOTION_FIELDS if self.has_motion else ()):
            setattr(self, name, torch.zeros((self.num_scenes, self.capacity) + tail, dtype=dtype, device=self.device))
        for name, dtype in K.TRACK_SCENE_FIELDS:
            setattr(self, name, torch.zeros((self.num_scenes,), dtype=dtype, device=self.device))
        self.xyz = self.feat = None

    def ensure_rows(self, xyz, feat):
        """allocates the bank rows from the first encode's (n, ...) outputs; later encodes must have the same row shapes"""
        if self.xyz is None:
            n = self.num_scenes * self.capacity
            self.xyz = torch.zeros((n,) + tuple(xyz.shape[1:]), dtype=xyz.dtype, device=self.device)
            self.feat = torch.zeros((n,) + tuple(feat.shape[1:]), dtype=feat.dtype, device=self.device)
        elif self.xyz.shape[1:] != xyz.shape[1:] or self.feat.shape[1:] != feat.shape[1:]:
            raise ValueError(f"encoder rows {tuple(xyz.shape[1:])} / {tuple(feat.shape[1:])} differ from the table's "
                             f"{tuple(self.xyz.shape[1:])} / {tuple(self.feat.shape[1:])}")

    def tracks(self, s):
        """-> (ids int64, labels, boxes (n, 7), ages, hits, rows int64 into xyz / feat) of scene s's alive slots, ascending slot
        order (reads the device: for inspection, not for the step)"""
        slot = self.alive[s].nonzero().squeeze(1)
        return (self.track_id[s, slot], self.label[s, slot], self.box[s, slot], self.age[s, slot], self.hits[s, slot],
                s * self.capacity + slot)

    def motion(self, s):
        """-> (box estimate (n, 7), velocity (n, 3) per unit of dt) of scene s's alive slots, ascending slot order, as tracks(s)
        lists them; after a step with motion the box estimate is the corrected one (reads the device: for inspection)"""
        if not self.has_motion:
            raise ValueError("this table keeps no motion state (TrackTable(..., motion=True))")
        slot = self.alive[s].nonzero().squeeze(1)
        return self.kf_box[s, slot], self.kf_vel[s, slot]

    def reset(self, s):
        """forgets every track of scene s: ids start again from 0"""
        for name, _, _ in K.TRACK_SLOT_FIELDS + (K.TRACK_MOTION_FIELDS if self.has_motion else ()):
            getattr(self, name)[s].zero_()
        for name, _ in K.TRACK_SCENE_FIELDS:
            getattr(self, name)[s] = 0


def _to_device(values, dtype, dev):
    t = torch.tensor(values, dtype=dtype)
    return t.pin_memory().to(dev, non_blocking=True) if dev.type == "cuda" else t


class MotionModel:
    """The constant-velocity Kalman filter a ReIDTracker keeps per track (include/pcreid.h, pcreid_track_predict), with
    AB3DMOT's settings as defaults.  State: the box (x, y, z, dx, dy, dz, yaw) and a velocity (vx, vy, vz) per unit of dt.
      init_var      initial variance of the 7 box values            q      process noise of the box values, per step
      init_vel_var  initial variance of the velocity                q_vel  process noise of the velocity, per step
      r             measurement noise of each box value
      gate_chi2     bound on the Mahalanobis distance of the predicted ground-plane centre to a detection's (chi-square,
                    2 degrees of freedom: 9.21 is the 99 % quantile); None: no such bound"""

    def __init__(self, init_var=10.0, init_vel_var=1e4, q=1.0, q_vel=0.01, r=1.0, gate_chi2=9.21):
        positive = ("init_var", "init_vel_var", "r", "gate_chi2")
        for name, v in dict(init_var=init_var, init_vel_var=init_vel_var, q=q, q_vel=q_vel, r=r, gate_chi2=gate_chi2).items():
            if v is None and name == "gate_chi2":
                setattr(self, name, None)
                continue
            v = float(v)
            if not math.isfinite(v) or v < 0 or (v == 0 and name in positive):
                raise ValueError(f"MotionModel.{name} must be finite and {'> 0' if name in positive else '>= 0'}; got {v}")
            setattr(self, name, v)

    def __repr__(self):
        return (f"MotionModel(init_var={self.init_var}, init_vel_var={self.init_vel_var}, q={self.q}, q_vel={self.q_vel}, "
                f"r={self.r}, gate_chi2={self.gate_chi2})")


class ReIDTracker:
    """A tracker over S scenes whose tracks live in a TrackTable: ids, ages, hits, retirement after ``max_age`` unmatched
    steps (None: never) and a bounded bank of ``capacity`` slots per scene, all updated on the device.

    ``step(frames, min_score, sample_ranks)`` runs, once each for all scenes: the segmented crop front-end, one encode, one
    gather of every active track's rows, kernels.track_gate_blocks (class_gate's rule, plus ``max_distance`` when given),
    the pair-list scorer (``'concat'`` models: scene by scene through their dense head), kernels.linear_assignment_blocks,
    kernels.track_update and kernels.track_scatter.  Its one host read is the S active counts.

    ``max_distance``: None, a float or one float per class; a track and a detection may then only be paired when their box
    centres are within that distance in the ground plane (x, y), tested in float32 as fl(dx*dx + dy*dy) <= fl(r*r).  That test
    is only meaningful when the boxes of every step are given in one fixed frame (e.g. world coordinates); the crop only needs
    each sweep and its boxes to agree.

    With max_age=None, a capacity that never fills and no max_distance, slots are handed out in append order and scene s's
    table is, row for row, the bank of PointReidentifier.step called with track_index = arange(len(bank)) and the stored
    labels; a detection's track id is then that bank row.

    ``motion``: None or a MotionModel.  With a model, the table keeps a Kalman filter per slot and the step runs
    kernels.track_predict (every active track of a scene with a frame, by that scene's ``dt``), then
    kernels.track_gate_motion_blocks instead of track_gate_blocks (``max_distance`` around the predicted centre, plus
    ``gate_chi2``), and kernels.track_correct after track_update (matched tracks take their detection, new tracks start with
    velocity 0): two launches more and no further host read.  A frozen scene is not predicted; pass the time elapsed since its
    last frame at its next one.  ``table.tracks(s)`` still gives the last matched boxes, ``table.motion(s)`` the filter's."""

    def __init__(self, model, num_scenes=1, capacity=1024, max_age=None, max_distance=None, replace_all=False, use_lengths=True,
                 num_classes=8, min_points=2, subsample_number=128, device="cuda", motion=None):
        if max_age is not None and max_age < 0:
            raise ValueError("max_age must be None or >= 0")
        if motion is not None and not isinstance(motion, MotionModel):
            raise TypeError("motion must be None or a MotionModel")
        self.model = model
        self.motion = motion
        self.table = TrackTable(num_scenes, capacity, replace_all, device, motion=motion is not None)
        self.max_age, self.use_lengths = max_age, use_lengths
        self.num_classes, self.min_points, self.subsample_number = num_classes, min_points, subsample_number
        self.radius_sq = None
        if max_distance is not None:
            r = torch.as_tensor(max_distance, dtype=torch.float32).flatten()
            if r.numel() == 1:
                r = r.expand(num_classes)
            if r.numel() != num_classes or bool((r < 0).any()) or bool(r.isnan().any()):
                raise ValueError(f"max_distance must be one non-negative float or {num_classes} of them")
            self.radius_sq = (r * r).contiguous().to(self.table.device)

    @torch.no_grad()
    def step(self, frames, min_score, sample_ranks=None, dt=1.0):
        """frames[s]: (sweep (P, >=3), bboxes (D_s, >=7), det_labels (D_s,)) or None (the scene is frozen: nothing ages);
        sample_ranks: None (drawn on the device) or one (D_s, N) int64 tensor per scene with a frame; dt: with a motion model,
        the time since each scene's previous frame, a float or one per scene (finite, >= 0; a frozen scene's entry is ignored).
        -> per scene (track_id_for_det (D_s,) int64, -1 for a detection that found no free slot; cost (A_s, D_s) logits, 0
        where not compared, or None when the scene had no active tracks), None for a frozen scene."""
        tab = self.table
        S, C, dev = tab.num_scenes, tab.capacity, tab.device
        if len(frames) != S:
            raise ValueError(f"{len(frames)} frames for {S} scenes")
        live = [s for s, f in enumerate(frames) if f is not None]
        results = [None] * S
        if not live:
            return results
        if sample_ranks is not None and any(sample_ranks[s] is None for s in live):
            raise ValueError("sample_ranks must give ranks for every scene with a frame, or be None")
        if self.motion is not None:
            dt = K.track_dt(dt, S, frozen=[s for s, f in enumerate(frames) if f is None])
        counts = tab.count.tolist()                                        # the step's one host read
        sweeps = [frames[s][0].float() for s in live]
        boxes = [frames[s][1][:, :7].float() for s in live]
        A, D = [0] * S, [0] * S
        for k, s in enumerate(live):
            A[s], D[s] = counts[s], boxes[k].shape[0]
        shapes = list(zip(A, D))
        # 1. crop / centre / resample every scene's detections from its own sweep; 2. one encode
        rank = None if sample_ranks is None else torch.cat([sample_ranks[s].to(sweeps[0].device, torch.int64) for s in live])
        det_points, det_len = crop_center_resample_scenes(torch.cat(boxes), torch.cat([w[:, :3] for w in sweeps]),
                                                          [D[s] for s in live], [w.shape[0] for w in sweeps],
                                                          self.subsample_number, sample_rank=rank)
        xyz_d, h_d = self.model.encode(det_points)
        tab.ensure_rows(xyz_d, h_d)
        det_label = torch.cat([frames[s][2] for s in live]).to(dev, torch.int32)
        det_length = det_len.to(dev, torch.int32)
        det_box = torch.cat(boxes).to(dev).contiguous()
        # 3. one gather of the rows of every scene's active tracks
        rows = tab.active.view(-1)[_to_device([s * C + i for s in range(S) for i in range(A[s])], torch.int64, dev)].long()
        xyz_t, h_t = tab.xyz[rows], tab.feat[rows]
        # 4. the gate of every scene's (A_s, D_s) block (with motion: on the predicted boxes)
        mm = self.motion
        if mm is None:
            gate = K.track_gate_blocks(tab, shapes, det_label, det_length, det_box, self.num_classes, self.min_points,
                                       self.use_lengths, self.radius_sq)
        else:
            K.track_predict(tab, shapes, dt, mm.q, mm.q_vel)
            gate = K.track_gate_motion_blocks(tab, shapes, det_label, det_length, det_box, self.num_classes, self.min_points,
                                              self.use_lengths, self.radius_sq, mm.r, mm.gate_chi2)
        d0, t0, e0 = [0], [0], [0]
        for a, d in shapes:
            d0.append(d0[-1] + d)
            t0.append(t0[-1] + a)
            e0.append(e0[-1] + a * d)
        # 5. the logits of the gated pairs
        if gate.numel() == 0:
            cost = torch.zeros((0,), device=dev, dtype=torch.float32)
        elif self.model.match_type == 'concat':
            cost = torch.cat([self.model.match_all_pairs(h_t[t0[s]:t0[s + 1]], xyz_t[t0[s]:t0[s + 1]], h_d[d0[s]:d0[s + 1]],
                                                         xyz_d[d0[s]:d0[s + 1]],
                                                         pair_mask=gate[e0[s]:e0[s + 1]].view(a, d)).reshape(-1)
                              for s, (a, d) in enumerate(shapes) if a * d])
        else:
            cost = score_pair_blocks(self.model, gate, shapes, d0[:-1], h_t, xyz_t, h_d, xyz_d)
        # 6. one assignment launch; 7. the table's bookkeeping; 8. the stored observations into their rows
        _, track_for_det = K.linear_assignment_blocks(cost, shapes, min_score, gate)
        det_track_id, det_row = K.track_update(tab, shapes, track_for_det, det_label, det_length, det_box, self.max_age,
                                               tab.replace_all)
        if mm is not None:
            K.track_correct(tab, shapes, rows, track_for_det, det_box, det_row, mm.init_var, mm.init_vel_var, mm.r)
        K.track_scatter(det_row, xyz_d, h_d, tab.xyz, tab.feat)
        for s in live:
            results[s] = (det_track_id[d0[s]:d0[s + 1]], cost[e0[s]:e0[s + 1]].view(A[s], D[s]) if A[s] else None)
        return results
