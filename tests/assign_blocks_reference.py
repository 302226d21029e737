"""kernels.linear_assignment_blocks's contract on the scipy oracle of tests/assign_reference.py, for tests that replace the
kernel on machines without a GPU."""
import numpy as np

from assign_reference import assign


def linear_assignment_blocks(score, shapes, min_score, pair_mask=None):
    """score 1-D torch float32 holding each (T_b, D_b) block row-major one after another, pair_mask bool packed the same way
    or None -> packed int64 (det_for_track (sum T_b,), track_for_det (sum D_b,)) on score's device."""
    import torch
    S = score.detach().cpu().numpy()
    M = None if pair_mask is None else pair_mask.cpu().numpy()
    d4t, t4d, e = [], [], 0
    for T, D in shapes:
        blk = S[e:e + T * D].reshape(T, D)
        r = assign(blk, np.float32(min_score), None if M is None else M[e:e + T * D].reshape(T, D))
        d4t.append(np.asarray(r[0], np.int64).reshape(T))
        t4d.append(np.asarray(r[1], np.int64).reshape(D))
        e += T * D
    cat = lambda parts: torch.from_numpy(np.concatenate(parts) if parts else np.zeros(0, np.int64)).to(score.device)
    return cat(d4t), cat(t4d)
