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
"""
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
        # 4. one match_pairs call over every scene's gated pairs, indices into the concatenated track / detection sets
        dev = gate.device
        e_off, t_off, d_off, cols = [0], [0], [], []
        for _, k, T, D in blocks:
            e_off.append(e_off[-1] + T * D)
            t_off.append(t_off[-1] + T)
            d_off.append(d0[k])
            cols.append(D)
        meta = torch.tensor([e_off[:-1], t_off[:-1], d_off, cols], dtype=torch.int64).to(dev)
        e = gate.nonzero().squeeze(1)
        blk = torch.searchsorted(torch.tensor(e_off[1:], dtype=torch.int64).to(dev), e, right=True)
        local = e - meta[0, blk]
        ti = meta[1, blk] + local // meta[3, blk]
        dj = meta[2, blk] + local % meta[3, blk]
        # 5. logits scattered into the packed cost
        cost = torch.zeros(gate.shape, device=dev, dtype=torch.float32)
        cost[e] = self.model.match_pairs(torch.cat(h_t), torch.cat(xyz_t), h_d, xyz_d, ti, dj)
        return cost, gate
