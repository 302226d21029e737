"""kernels.track_gate_blocks / track_update / track_scatter restated in plain torch / numpy on the CPU, straight from the track
table's policy (include/pcreid.h, models/tracking.py TrackTable).  Same signatures as the kernel wrappers, so tests can put them
in their place on machines without a GPU; the GPU tests compare the kernels against them.  ``table`` is any object with the
tensors of kernels.TRACK_SLOT_FIELDS / TRACK_SCENE_FIELDS, here on the CPU."""
import numpy as np
import torch


def track_gate_blocks(table, shapes, det_label, det_length, det_box, num_classes=8, min_points=2, use_lengths=True,
                      radius_sq=None):
    """-> bool (sum A_s * D_s,): scene s's row-major (A_s, D_s) gate after scene s-1's"""
    parts, d0 = [], 0
    for s, (A, D) in enumerate(shapes):
        rows = table.active[s, :A].long()
        lt, ln, bt = table.label.view(-1)[rows], table.length.view(-1)[rows], table.box.view(-1, 7)[rows]
        ld, lnd, bd = det_label[d0:d0 + D], det_length[d0:d0 + D], det_box[d0:d0 + D]
        ok_t = (lt >= 0) & (lt < num_classes)
        ok_d = (ld >= 0) & (ld < num_classes)
        if use_lengths:
            ok_t = ok_t & (ln >= min_points)
            ok_d = ok_d & (lnd >= min_points)
        g = (lt[:, None] == ld[None, :]) & ok_t[:, None] & ok_d[None, :]
        if radius_sq is not None:
            dx = bt[:, None, 0] - bd[None, :, 0]            # float32, one rounding per operation
            dy = bt[:, None, 1] - bd[None, :, 1]
            r2 = radius_sq[lt.clamp(0, num_classes - 1).long()]
            g = g & ((dx * dx + dy * dy) <= r2[:, None])
        parts.append(g.reshape(-1))
        d0 += D
    return torch.cat(parts) if parts else torch.zeros((0,), dtype=torch.bool)


def track_update(table, shapes, track_for_det, det_label, det_length, det_box, max_age=None, replace_all=False):
    """updates table in place -> (det_track_id int64, det_row int32) over the packed detections"""
    S, C = table.alive.shape
    alive, tid, label = table.alive.view(-1).numpy(), table.track_id.view(-1).numpy(), table.label.view(-1).numpy()
    length, age, hits = table.length.view(-1).numpy(), table.age.view(-1).numpy(), table.hits.view(-1).numpy()
    box, active = table.box.view(-1, 7).numpy(), table.active.numpy()
    next_id, dropped, count = table.next_id.numpy(), table.dropped.numpy(), table.count.numpy()
    tfd_all, dl, dn, db = track_for_det.numpy(), det_label.numpy(), det_length.numpy(), det_box.numpy()
    n = sum(d for _, d in shapes)
    det_track_id = np.full(n, -1, np.int64)
    det_row = np.full(n, -1, np.int32)
    d0 = 0
    for s, (A, D) in enumerate(shapes):
        act = [int(r) for r in active[s, :A]]
        tfd = [int(t) for t in tfd_all[d0:d0 + D]]
        # 1. matched
        matched = set()
        for d, t in enumerate(tfd):
            if t < 0:
                continue
            matched.add(t)
            r, j = act[t], d0 + d
            age[r], hits[r], box[r] = 0, hits[r] + 1, db[j]
            if replace_all or length[r] <= dn[j]:
                length[r], det_row[j] = dn[j], r
            det_track_id[j] = tid[r]
        # 2. unmatched active tracks
        for i, r in enumerate(act):
            if i not in matched:
                age[r] += 1
                if max_age is not None and age[r] > max_age:
                    alive[r] = False
        # 3. unmatched detections into the lowest free slots
        free = [s * C + c for c in range(C) if not alive[s * C + c]]
        first, k = int(next_id[s]), 0
        for d, t in enumerate(tfd):
            if t >= 0:
                continue
            j = d0 + d
            if k < len(free):
                r = free[k]
                alive[r], tid[r], label[r], length[r], age[r], hits[r], box[r] = True, first + k, dl[j], dn[j], 0, 1, db[j]
                det_track_id[j], det_row[j] = first + k, r
            k += 1
        stored = min(k, len(free))
        next_id[s], dropped[s] = first + stored, dropped[s] + k - stored
        # 4. the next active list (entries past the count are left as they were)
        if A or D:
            rows = [s * C + c for c in range(C) if alive[s * C + c]]
            active[s, :len(rows)] = rows
            count[s] = len(rows)
        d0 += D
    return torch.from_numpy(det_track_id), torch.from_numpy(det_row)


def track_scatter(det_row, det_xyz, det_feat, xyz, feat):
    keep = (det_row >= 0).nonzero().squeeze(1)
    rows = det_row[keep].long()
    xyz[rows] = det_xyz[keep]
    feat[rows] = det_feat[keep]
