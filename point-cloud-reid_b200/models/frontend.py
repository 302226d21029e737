"""Crop -> centre -> resample front-end: one LiDAR sweep + boxes -> the (B, N, 3) encoder input.

Mirrors the deprecated tracker's ``interpolate_per_frame`` + ``get_input_batch``
(mmdet3d/models/trackers/deprecated/pc_utils.py:31-96): points inside each box (DepthInstance3DBoxes with origin
(0.5, 0.5, 0.5), core/bbox/structures/depth_box3d.py:256-282), expressed in the box frame (inverse of the box pose),
resampled WITH replacement to ``subsample_number`` points; boxes without points give zeros.  The reference builds a (P, B)
mask, B python crops, a padded (B, Lmax, 3) batch and its homogeneous copy; here two kernels (csrc/frontend.cu) go from
the sweep to the encoder input through a bit mask."""
import torch

from .. import _lib
from .. import torch_ops as _T

_OPS = _T.ops


def points_in_boxes_mask(bboxes, pts):
    """-> (mask (B, ntiles, 32) int32 bit mask, counts (B, ntiles) int32, lengths (B,) int64)."""
    if not (bboxes.is_cuda and pts.is_cuda):
        raise RuntimeError("pcreid_b200 kernels need CUDA tensors (there is no CPU fallback)")
    assert bboxes.dtype == torch.float32 and pts.dtype == torch.float32 and bboxes.shape[1] == 7
    bboxes, pts = bboxes.contiguous(), pts.contiguous()
    P, B = pts.shape[0], bboxes.shape[0]
    L = _lib.lib()
    nt = L.pcreid_crop_tiles(P)
    mask = torch.empty((B, nt, 32), device=pts.device, dtype=torch.int32)
    counts = torch.empty((B, nt), device=pts.device, dtype=torch.int32)
    _OPS.crop_mask(P, B, pts, pts.shape[1], bboxes, mask, counts)
    return mask, counts, counts.sum(1, dtype=torch.int64)


def crop_center_resample(bboxes, pts, subsample_number, sample_rank=None, generator=None):
    """bboxes (B, 7) = (x, y, z centre, dx, dy, dz, yaw), pts (P, >=3) -> (out (1, B, N, 3), lengths (1, B)).

    ``sample_rank`` (B, N) int64: which in-box point (in point order) each output slot takes -- what the reference draws with
    ``torch.randint(high=length)`` per box (pc_utils.py:84-85).  When omitted, ranks are drawn on the device as
    floor(U[0,1) * length): the same distribution, not the reference's host random stream."""
    P, B, N = pts.shape[0], bboxes.shape[0], int(subsample_number)
    if P == 0 or B == 0:        # empty sweep / no boxes: zero crops with zero lengths, as the reference returns (pc_utils.py:88-92)
        if not (bboxes.is_cuda and pts.is_cuda):
            raise RuntimeError("pcreid_b200 kernels need CUDA tensors (there is no CPU fallback)")
        return (torch.zeros((1, B, N, 3), device=pts.device, dtype=torch.float32),
                torch.zeros((1, B), device=pts.device, dtype=torch.int64))
    mask, counts, lengths = points_in_boxes_mask(bboxes, pts)
    bboxes, pts = bboxes.contiguous(), pts.contiguous()
    prefix = torch.zeros((B, counts.shape[1] + 1), device=pts.device, dtype=torch.int32)
    prefix[:, 1:] = torch.cumsum(counts, 1, dtype=torch.int32)
    if sample_rank is None:
        u = torch.rand((B, N), device=pts.device, generator=generator)
        sample_rank = (u * lengths[:, None]).long()
    sample_rank = sample_rank.to(device=pts.device, dtype=torch.int64).contiguous()
    assert sample_rank.shape == (B, N)
    out = torch.empty((B, N, 3), device=pts.device, dtype=torch.float32)
    _OPS.crop_gather(P, B, N, pts, pts.shape[1], bboxes, mask, prefix, sample_rank, out)
    return out.unsqueeze(0), lengths.unsqueeze(0)


def _to_device_async(host, dtype, device):
    """host list -> device tensor through pinned memory: an asynchronous copy, no synchronisation with the device."""
    t = torch.tensor(host, dtype=dtype)
    return t.pin_memory().to(device, non_blocking=True) if torch.device(device).type == "cuda" else t.to(device)


def crop_center_resample_scenes(bboxes, pts, box_counts, point_counts, subsample_number, sample_rank=None):
    """crop_center_resample over S sweeps in one launch per pass (pcreid_crop_mask_scenes / pcreid_crop_gather_scenes).
    pts (sum P_s, >=3) = the sweeps one after another, bboxes (sum B_s, 7) = each scene's boxes one after another; box_counts /
    point_counts: host sequences of B_s / P_s.  Each box is cropped from its own sweep only.
    -> (out (sum B_s, N, 3), lengths (sum B_s,) int64).  With ``sample_rank`` (sum B_s, N) int64 given, scene s's rows equal
    crop_center_resample on that scene with its rows of sample_rank; without it, ranks are drawn on the device (the same
    distribution, not the same draws)."""
    if not (bboxes.is_cuda and pts.is_cuda):
        raise RuntimeError("pcreid_b200 kernels need CUDA tensors (there is no CPU fallback)")
    box_counts, point_counts = [int(b) for b in box_counts], [int(p) for p in point_counts]
    S, N, dev = len(box_counts), int(subsample_number), pts.device
    if len(point_counts) != S or min(box_counts + point_counts, default=0) < 0:
        raise ValueError("box_counts and point_counts must hold one non-negative size per scene")
    if bboxes.dtype != torch.float32 or pts.dtype != torch.float32 or bboxes.dim() != 2 or bboxes.shape[1] != 7:
        raise ValueError("bboxes must be float32 (sum B_s, 7) and pts float32 (sum P_s, >=3)")
    if pts.dim() != 2 or pts.shape[1] < 3:
        raise ValueError("pts must be (sum P_s, >=3)")
    if bboxes.shape[0] != sum(box_counts) or pts.shape[0] != sum(point_counts):
        raise ValueError("bboxes / pts rows must be the sums of box_counts / point_counts")
    B = bboxes.shape[0]
    L = _lib.lib()
    nt = [L.pcreid_crop_tiles(p) for p in point_counts]
    offs = [[0] for _ in range(4)]
    for p, b, t in zip(point_counts, box_counts, nt):
        for row, v in zip(offs, (p, b, t, b * t)):
            row.append(row[-1] + v)
    C = offs[3][-1]
    if C * 32 >= 1 << 31:
        raise ValueError("mask of the segmented front-end exceeds 2^31 words: split the scenes over several calls")
    off = _to_device_async(offs, torch.int32, dev)
    bboxes, pts = bboxes.contiguous(), pts.contiguous()
    mask = torch.empty((C, 32), device=dev, dtype=torch.int32)
    counts = torch.empty((C,), device=dev, dtype=torch.int32)
    if C > 0:                   # else no box has a tile: every crop is empty
        _OPS.crop_mask_scenes(S, offs[2][-1], max(box_counts), pts, pts.shape[1], bboxes, off, mask, counts)
    # per box: its ntiles count words, and its prefix (ntiles + 1) at count word + global box index
    nt_box = _to_device_async([t for b, t in zip(box_counts, nt) for _ in range(b)], torch.int64, dev)
    seg = torch.repeat_interleave(torch.arange(B, device=dev), nt_box, output_size=C)
    incl = counts.cumsum(0, dtype=torch.int64)
    start = torch.cumsum(nt_box, 0) - nt_box                                  # first count word of each box
    within = incl - (incl - counts)[start[seg]]                             # inclusive scan inside each box
    prefix = torch.zeros((B + C,), device=dev, dtype=torch.int32)
    prefix[torch.arange(C, device=dev) + seg + 1] = within.to(torch.int32)
    lengths = torch.zeros((B,), device=dev, dtype=torch.int64).index_add_(0, seg, counts.to(torch.int64))
    if sample_rank is None:
        sample_rank = (torch.rand((B, N), device=dev) * lengths[:, None]).long()
    sample_rank = sample_rank.to(device=dev, dtype=torch.int64).contiguous()
    if sample_rank.shape != (B, N):
        raise ValueError(f"sample_rank must be ({B}, {N})")
    out = torch.empty((B, N, 3), device=dev, dtype=torch.float32)
    _OPS.crop_gather_scenes(S, B, N, pts, pts.shape[1], bboxes, off, mask, prefix, sample_rank, out)
    return out, lengths
