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
"""
import torch

from .. import kernels as K
from .frontend import crop_center_resample


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
