"""kernels.track_predict / track_correct / track_gate_motion_blocks restated in torch on the CPU, in the operation order
include/pcreid.h pins (one rounding per operation, nothing fused), with the wrappers' signatures: tests put them in the
kernels' place on machines without a GPU, and the GPU tests compare the kernels against them bit for bit.  ``table`` is any
object with the tensors of kernels.TRACK_SLOT_FIELDS / TRACK_MOTION_FIELDS; the arithmetic runs in the dtype of its motion
fields (float32 as on the device, or float64 to compare the compact filter with the textbook one)."""
import math
import types

import torch

import track_table_reference as TT


def _c(v, dtype):
    return torch.tensor(v, dtype=torch.float32).to(dtype)         # a scalar as the kernel receives it (f32), in dtype


def _pi(dtype):
    return torch.tensor(math.pi, dtype=dtype)


def wrap(a):
    two_pi = 2 * _pi(a.dtype)                                        # fl(2 pi) = 2 fl(pi)
    return a - two_pi * torch.round(a / two_pi)                      # round: to nearest even, as rintf


def _packed_rows(table, shapes):
    return torch.cat([table.active[s, :a].long() for s, (a, _) in enumerate(shapes)] + [torch.zeros(0, dtype=torch.long)])


def track_predict(table, shapes, dt, q=1.0, q_vel=0.01):
    S = len(shapes)
    dt = [dt] * S if isinstance(dt, (int, float)) else list(dt)
    dtype = table.kf_box.dtype
    rows = _packed_rows(table, shapes)
    dts = torch.cat([_c(float(dt[s]), dtype).expand(a) for s, (a, _) in enumerate(shapes)] + [torch.zeros(0, dtype=dtype)])
    q, q_vel = _c(q, dtype), _c(q_vel, dtype)
    box, vel, cov = table.kf_box.view(-1, 7), table.kf_vel.view(-1, 3), table.kf_cov.view(-1, 13)
    b, v, P = box[rows], vel[rows], cov[rows]
    for a in range(3):
        pp, pv, vv = P[:, 3 * a].clone(), P[:, 3 * a + 1].clone(), P[:, 3 * a + 2].clone()
        b[:, a] = b[:, a] + dts * v[:, a]
        t = pv + dts * vv
        P[:, 3 * a] = (pp + dts * (pv + t)) + q
        P[:, 3 * a + 1] = t
        P[:, 3 * a + 2] = vv + q_vel
    P[:, 9:] = P[:, 9:] + q
    box[rows], cov[rows] = b, P


def track_correct(table, shapes, track_rows, track_for_det, det_box, det_row, init_var=10.0, init_vel_var=1e4, r=1.0):
    dtype = table.kf_box.dtype
    box, vel, cov = table.kf_box.view(-1, 7), table.kf_vel.view(-1, 3), table.kf_cov.view(-1, 13)
    t0 = torch.tensor([0] + [a for a, _ in shapes], dtype=torch.long).cumsum(0)[:-1]
    t_first = torch.repeat_interleave(t0, torch.tensor([d for _, d in shapes], dtype=torch.long))
    z_all = det_box.to(dtype)
    # births: box (yaw wrapped), velocity 0, the initial covariance
    born = ((track_for_det < 0) & (det_row >= 0)).nonzero().squeeze(1)
    br = det_row[born].long()
    zb = z_all[born].clone()
    zb[:, 6] = wrap(zb[:, 6])
    box[br], vel[br] = zb, torch.zeros((born.numel(), 3), dtype=dtype)
    P0 = torch.tensor([init_var, 0.0, init_vel_var] * 3 + [init_var] * 4, dtype=torch.float32).to(dtype)
    cov[br] = P0.expand(born.numel(), 13)
    # matched: the update of each axis
    m = (track_for_det >= 0).nonzero().squeeze(1)
    rows = track_rows[t_first[m] + track_for_det[m]].long()
    z, b, v, P = z_all[m], box[rows], vel[rows], cov[rows]
    r = _c(r, dtype)
    for a in range(3):
        pp, pv, vv = P[:, 3 * a].clone(), P[:, 3 * a + 1].clone(), P[:, 3 * a + 2].clone()
        s = pp + r
        kp, kv = pp / s, pv / s
        y = z[:, a] - b[:, a]
        b[:, a] = b[:, a] + kp * y
        v[:, a] = v[:, a] + kv * y
        P[:, 3 * a + 2] = vv - kv * pv
        P[:, 3 * a + 1] = kv * r
        P[:, 3 * a] = kp * r
    for a in range(3, 6):
        k = P[:, 6 + a] / (P[:, 6 + a] + r)
        b[:, a] = b[:, a] + k * (z[:, a] - b[:, a])
        P[:, 6 + a] = k * r
    k = P[:, 12] / (P[:, 12] + r)
    y = wrap(z[:, 6] - b[:, 6])
    y = torch.where(y.abs() > _pi(dtype) / 2, wrap(y + _pi(dtype)), y)
    b[:, 6] = wrap(b[:, 6] + k * y)
    P[:, 12] = k * r
    box[rows], vel[rows], cov[rows] = b, v, P


def track_gate_motion_blocks(table, shapes, det_label, det_length, det_box, num_classes=8, min_points=2, use_lengths=True,
                             radius_sq=None, r=1.0, gate_chi2=None):
    predicted = types.SimpleNamespace(active=table.active, label=table.label, length=table.length, box=table.kf_box)
    gate = TT.track_gate_blocks(predicted, shapes, det_label, det_length, det_box, num_classes, min_points, use_lengths,
                                radius_sq)
    if gate_chi2 is None:
        return gate
    parts, d0 = [], 0
    r, chi2 = _c(r, torch.float32), _c(gate_chi2, torch.float32)
    for s, (A, D) in enumerate(shapes):
        rows = table.active[s, :A].long()
        bt, P, bd = table.kf_box.view(-1, 7)[rows], table.kf_cov.view(-1, 13)[rows], det_box[d0:d0 + D]
        dx = bt[:, None, 0] - bd[None, :, 0]
        dy = bt[:, None, 1] - bd[None, :, 1]
        sx, sy = (P[:, 0] + r)[:, None], (P[:, 3] + r)[:, None]
        parts.append(((dx * dx / sx + dy * dy / sy) <= chi2).reshape(-1))
        d0 += D
    return gate & torch.cat(parts + [torch.zeros(0, dtype=torch.bool)])
