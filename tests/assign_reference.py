"""CPU oracle of the gated linear assignment (include/pcreid.h, pcreid_lsap), in float64 on scipy.

A pair (t, d) is admissible when mask[t, d], S[t, d] is finite and S[t, d] > tau (strictly); its weight is
w = double(S) - double(tau).  The answer is a matching of admissible pairs of maximum total weight.  scipy solves it as the
T x (D + T) min-cost assignment C with C[t, d] = -w (admissible) or +inf, C[t, D + t] = 0 ("leave t unmatched") and every
other dummy entry +inf; C is always feasible.  `brute_force_value` enumerates every matching and checks that reduction."""
import itertools

import numpy as np
from scipy.optimize import linear_sum_assignment


def admissible(score, tau, mask=None):
    S = np.asarray(score, dtype=np.float32)
    ok = np.isfinite(S) & (S > np.float32(tau))
    return ok if mask is None else ok & np.asarray(mask, dtype=bool)


def weights(score, tau):
    with np.errstate(invalid="ignore"):
        return np.asarray(score, dtype=np.float32).astype(np.float64) - np.float64(np.float32(tau))


def assign(score, tau, mask=None):
    """score (T, D) float32, tau a float32 value, mask (T, D) bool or None -> (det_for_track (T,), track_for_det (D,)) int64,
    -1 for unmatched."""
    S = np.asarray(score, dtype=np.float32)
    T, D = S.shape
    adm = admissible(S, tau, mask)
    C = np.full((T, D + T), np.inf)
    C[:, :D] = np.where(adm, -weights(S, tau), np.inf)
    C[np.arange(T), D + np.arange(T)] = 0.0
    d4t, t4d = np.full(T, -1, np.int64), np.full(D, -1, np.int64)
    if T == 0:
        return d4t, t4d
    rows, cols = linear_sum_assignment(C)
    for t, d in zip(rows, cols):
        if d < D:
            d4t[t], t4d[d] = d, t
    return d4t, t4d


def objective(score, tau, det_for_track, mask=None):
    """total weight of a matching; raises if it uses an inadmissible pair or a detection twice."""
    adm, W = admissible(score, tau, mask), weights(score, tau)
    d4t = np.asarray(det_for_track)
    used = d4t[d4t >= 0]
    if len(set(used.tolist())) != used.size:
        raise AssertionError("a detection is matched twice")
    total = 0.0
    for t, d in enumerate(d4t):
        if d >= 0:
            if not adm[t, d]:
                raise AssertionError(f"inadmissible pair ({t}, {d}) matched")
            total += W[t, d]
    return total


def consistent(det_for_track, track_for_det):
    """the two output vectors describe the same matching."""
    d4t, t4d = np.asarray(det_for_track), np.asarray(track_for_det)
    return (all(t4d[d] == t for t, d in enumerate(d4t) if d >= 0)
            and all(d4t[t] == d for d, t in enumerate(t4d) if t >= 0))


def brute_force_value(score, tau, mask=None):
    """maximum total weight over every matching of admissible pairs (small T, D only)."""
    adm, W = admissible(score, tau, mask), weights(score, tau)
    T, D = adm.shape
    best = 0.0
    for k in range(1, min(T, D) + 1):
        for rows in itertools.combinations(range(T), k):
            for cols in itertools.permutations(range(D), k):
                if all(adm[t, d] for t, d in zip(rows, cols)):
                    best = max(best, sum(W[t, d] for t, d in zip(rows, cols)))
    return best


def linear_assignment(score, min_score, pair_mask=None):
    """kernels.linear_assignment's contract on the oracle, for tests that replace the kernel on machines without a GPU:
    score (T, D) or (B, T, D) torch float32, pair_mask bool or None -> int64 (det_for_track, track_for_det) on score's device."""
    import torch
    S = score.detach().cpu().numpy()
    M = None if pair_mask is None else pair_mask.cpu().numpy()
    batched = S.ndim == 3
    if not batched:
        S, M = S[None], (None if M is None else M[None])
    res = [assign(S[b], np.float32(min_score), None if M is None else M[b]) for b in range(S.shape[0])]
    d4t = torch.from_numpy(np.stack([r[0] for r in res]).reshape(S.shape[0], S.shape[1])).to(score.device)
    t4d = torch.from_numpy(np.stack([r[1] for r in res]).reshape(S.shape[0], S.shape[2])).to(score.device)
    return (d4t, t4d) if batched else (d4t[0], t4d[0])
