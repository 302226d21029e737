"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the crop -> centre -> resample front-end of the deprecated tracker.

Follows, line by line:
  mmdet3d/models/trackers/deprecated/pc_utils.py:31-76  interpolate_per_frame  (crop, inverse box pose)
  mmdet3d/models/trackers/deprecated/pc_utils.py:80-96  get_input_batch        (resample with replacement, zeros if empty)
  mmdet3d/core/bbox/structures/base_box3d.py:61-64      origin (0.5,0.5,0.5) -> bottom centre
  mmdet3d/core/bbox/structures/depth_box3d.py:256-282   depth -> LiDAR frame for points and boxes
  mmdet3d/core/bbox/structures/box_3d_mode.py:125-148   DEPTH -> LIDAR box conversion (rt_mat, size swap)
  mmdet3d/ops/roiaware_pool3d/src/points_in_boxes_cuda.cu:24-49, 79-105   the in-box test
PINNED (tests/test_frontend_pinned.py, wherever PCREID_REFERENCE_ROOT names the upstream source tree) against the reference's own pc_utils.py and
core/bbox/structures/*.py imported unmodified by path (oracle/ref_loader.load_frontend): box origin / frame conversion and
crop order exactly, centred coordinates within 2e-5 (fp32 torch there, fp64 numpy here), sampling with the same torch.randint
draws.  Stand-ins there: pytorch3d (absent; Pointclouds.points_padded and axis_angle_to_matrix restated from pytorch3d 0.7)
and the compiled points_in_boxes_batch op (-> pib_kernel_lidar below, which is pinned on the GPU box against the
reference's own points_in_boxes_cuda.cu when oracle/_ref/libref_pib.so could be built)."""
import ctypes
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
f32, f64 = np.float32, np.float64


def pib_kernel_lidar(boxes_lidar, pts_lidar):
    """points_in_boxes_cuda.cu:24-49, 79-105 (check_pt_in_box3d + lidar_to_local_coords) on boxes (T, 7) = (x, y, z_bottom, w, l,
    h, rz) and points (M, 3), both already in the LiDAR frame -> (inside bool (T, M), margin (T, M))."""
    b = np.asarray(boxes_lidar, f32)
    p = np.asarray(pts_lidar, f32)
    cx, cy, zb, w, l, h, rz = (b[:, i] for i in range(7))
    xl, yl, zl = p[:, 0], p[:, 1], p[:, 2]
    hh = h.astype(f64) / 2.0
    cz = (zb.astype(f64) + hh).astype(f32)                                  # points_in_boxes_cuda.cu:42
    dz = np.abs((zl[None, :] - cz[:, None]).astype(f32)).astype(f64)
    ang = (rz.astype(f64) + np.pi / 2).astype(f32)                          # :28
    c, s = np.cos(ang).astype(f32), np.sin(ang).astype(f32)
    sx = (xl[None, :] - cx[:, None]).astype(f32)
    sy = (yl[None, :] - cy[:, None]).astype(f32)
    # nvcc contraction of the reference expressions (SASS): lx = fma(sx, c, -(sy*s)), ly = fma(sy, c, sx*s)
    lx = (sx.astype(f64) * c[:, None].astype(f64) - (sy * s[:, None]).astype(f32).astype(f64)).astype(f32)
    ly = (sy.astype(f64) * c[:, None].astype(f64) + (sx * s[:, None]).astype(f32).astype(f64)).astype(f32)
    hl, hw = l.astype(f64) / 2.0, w.astype(f64) / 2.0
    inside = (dz <= hh[:, None]) & (lx > -hl[:, None]) & (lx < hl[:, None]) & (ly > -hw[:, None]) & (ly < hw[:, None])
    margin = np.minimum(np.minimum(np.abs(hh[:, None] - dz), np.abs(hl[:, None] - np.abs(lx))), np.abs(hw[:, None] - np.abs(ly)))
    return inside, margin


def depth_boxes_to_lidar(bboxes):
    """DepthInstance3DBoxes(bboxes, origin=(0.5, 0.5, 0.5)).convert_to(LIDAR).tensor (base_box3d.py:61-64,
    box_3d_mode.py:125-148): (x, y, z_centre, dx, dy, dz, yaw) -> (y, -x, z_bottom, dy, dx, dz, yaw)."""
    b = np.asarray(bboxes, f32)
    zb = (b[:, 2] + b[:, 5] * f32(-0.5)).astype(f32)                       # base_box3d.py:61-64
    return np.stack([b[:, 1], -b[:, 0], zb, b[:, 4], b[:, 3], b[:, 5], b[:, 6]], 1).astype(f32)


def points_in_boxes(bboxes, pts):
    """-> bool (B, P), plus the margin (B, P) = distance of the decisive coordinate to the nearest box face (for
    margin-aware comparisons: cosf / sinf differ in the last bit between libm and CUDA)."""
    p = np.asarray(pts, f32)[:, :3]
    pl = np.stack([p[:, 1], -p[:, 0], p[:, 2]], 1)                          # depth_box3d.py:270-272
    return pib_kernel_lidar(depth_boxes_to_lidar(bboxes), pl)


def crop_center_resample(bboxes, pts, subsample_number, sample_rank, inside=None):
    """-> (out (1, B, N, 3) float32, lengths (1, B) int64); sample_rank (B, N) as drawn by get_input_batch's randint."""
    b = np.asarray(bboxes, f32)
    p = np.asarray(pts, f32)[:, :3]
    if inside is None:
        inside, _ = points_in_boxes(b, p)
    B, N = b.shape[0], int(subsample_number)
    out = np.zeros((1, B, N, 3), f32)
    lengths = inside.sum(1).astype(np.int64)
    for i in range(B):
        if lengths[i] == 0:
            continue                                                        # pc_utils.py:84, 89: zeros
        crop = p[inside[i]]                                                 # point order (pc_utils.py:50)
        yaw = float(b[i, 6])
        c, s = np.cos(yaw), np.sin(yaw)
        A = np.eye(4)                                                       # get_affine_torch(rotation=-(0,0,yaw)) -> Rz(-yaw)
        A[:3, :3] = np.array([[c, s, 0.0], [-s, c, 0.0], [0.0, 0.0, 1.0]])
        A[:3, 3] = b[i, :3]
        Ainv = np.linalg.inv(A)                                             # inverse=True
        hom = np.concatenate([crop.astype(f64), np.ones((crop.shape[0], 1))], 1)
        centered = (Ainv @ hom.T).T[:, :3]
        out[0, i] = centered[np.asarray(sample_rank[i], np.int64)].astype(f32)
    return torch.from_numpy(out), torch.from_numpy(lengths[None])


def ref_pib_available():
    return os.path.exists(os.path.join(_HERE, "_ref", "libref_pib.so")) and torch.cuda.is_available()


def ref_points_in_boxes_lidar(boxes_lidar, pts_lidar):
    """the reference's points_in_boxes_batch_launcher on the GPU: boxes (1, T, 7) / points (1, M, 3) in the LiDAR frame
    -> int32 (1, M, T).  (Launches on the default stream, as the reference does.)"""
    L = ctypes.CDLL(os.path.join(_HERE, "_ref", "libref_pib.so"))
    Bt, T, _ = boxes_lidar.shape
    M = pts_lidar.shape[1]
    out = torch.zeros((Bt, M, T), dtype=torch.int32, device=pts_lidar.device)
    torch.cuda.synchronize()
    L.ref_points_in_boxes_batch(Bt, T, M, ctypes.c_void_p(boxes_lidar.data_ptr()), ctypes.c_void_p(pts_lidar.data_ptr()),
                                ctypes.c_void_p(out.data_ptr()))
    torch.cuda.synchronize()
    return out
