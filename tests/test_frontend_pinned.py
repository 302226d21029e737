"""Pins oracle/frontend_oracle.py (crop -> centre -> resample, SURVEY 8f row 2) to the reference's OWN code:
models/trackers/deprecated/pc_utils.py (interpolate_per_frame, get_input_batch) and core/bbox/structures/*.py
(DepthInstance3DBoxes, Box3DMode.convert) imported unmodified by path (oracle/ref_loader.load_frontend) and run on CPU; pytorch3d
and the compiled points_in_boxes op are stand-ins (see the loader).  Runs where PCREID_REFERENCE_ROOT names the upstream source tree."""
import numpy as np
import pytest
import torch

from oracle import frontend_oracle as FO
from oracle import ref_loader

pytestmark = pytest.mark.skipif(not ref_loader.frontend_available(), reason=ref_loader.MISSING)


@pytest.fixture(scope="module")
def R():
    return ref_loader.load_frontend()


def _scene(seed, P=6000, B=14):
    g = torch.Generator().manual_seed(seed)
    pts = (torch.rand(P, 4, generator=g) - 0.5) * torch.tensor([40., 40., 4., 1.])
    boxes = torch.cat([(torch.rand(B, 3, generator=g) - 0.5) * torch.tensor([30., 30., 2.]), 1.5 + 3 * torch.rand(B, 3, generator=g),
                       (torch.rand(B, 1, generator=g) - 0.5) * 6.28], 1).float()
    boxes[0, :3] = torch.tensor([500., 500., 0.])          # a box without points: zero-filled crop (pc_utils.py:84, 89)
    return boxes, pts.float()


@pytest.mark.parametrize("seed", [0, 1])
def test_box_conversion_and_in_box_mask_vs_reference(R, seed):
    boxes, pts = _scene(seed)
    lb = R.DepthInstance3DBoxes(boxes, origin=(0.5, 0.5, 0.5))
    assert np.array_equal(lb.convert_to(R.Box3DMode.LIDAR).tensor.numpy(), FO.depth_boxes_to_lidar(boxes.numpy()))
    ref = lb.points_in_boxes(pts[:, :3].unsqueeze(0)).numpy().T.astype(bool)          # (B, P)
    ins, _ = FO.points_in_boxes(boxes.numpy(), pts.numpy())
    assert np.array_equal(ref, ins) and ins[0].sum() == 0 and ins.sum() > 100


@pytest.mark.parametrize("seed,n", [(0, 64), (1, 128)])
def test_crop_center_resample_vs_reference(R, seed, n):
    boxes, pts = _scene(seed)
    centered, lengths = R.interpolate_per_frame(boxes, pts, 'cpu')
    torch.manual_seed(5)
    ref = R.get_input_batch(centered, lengths, n, 'cpu')
    torch.manual_seed(5)              # the same draws get_input_batch makes (pc_utils.py:84-86), handed to the oracle as ranks
    ranks = torch.cat([torch.randint(high=int(x), size=(1, n)) if x != 0 else torch.zeros((1, n)) for x in lengths.reshape(-1)]).long()
    out, lens = FO.crop_center_resample(boxes.numpy(), pts.numpy(), n, ranks.numpy())
    assert torch.equal(lens, lengths) and ref.shape == out.shape == (1, boxes.shape[0], n, 3)
    assert (ref - out).abs().max() < 2e-5 and (out[0, 0] == 0).all()
