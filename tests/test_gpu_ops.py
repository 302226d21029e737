"""-m gpu: the five mmdet3d point ops + the torch-path kNNs, through the C ABI, bit-exact against
  (a) the C restatement of the reference kernels (oracle/ops_oracle.c) and
  (b) the reference's own .cu files compiled unmodified for sm_100a (oracle/_ref), when that library travelled."""
import pytest
import torch

from oracle import ops_oracle as P
from oracle import reid_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"


def clouds(B, N, seed, kind):
    if kind == "free":
        return O.synth_objects(B, N, seed)
    if kind == "dup":
        return O.synth_objects(B, N, seed, dup=True)
    if kind == "same":            # all points identical (subsamplePC of a <=2 point object, datasets/utils.py:610-619)
        return O.synth_objects(B, 1, seed).expand(B, N, 3).contiguous()
    if kind == "zero":
        return torch.zeros(B, N, 3)
    if kind == "u3":              # three unique points
        base = O.synth_objects(B, 3, seed)
        pick = torch.randint(0, 3, (B, N), generator=torch.Generator().manual_seed(seed))
        return torch.gather(base, 1, pick.unsqueeze(-1).expand(B, N, 3)).contiguous()
    raise ValueError(kind)


KINDS = ["free", "dup", "same", "zero", "u3"]


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N,M", [(256, 128), (160, 80), (1000, 64), (37, 37), (2048, 16), (5000, 8)])
def test_fps_bit_exact(kind, N, M):
    from pcreid_b200.ops import furthest_point_sample
    x = clouds(3, N, 1, kind)
    got = furthest_point_sample(x.to(DEV), M).cpu()
    assert got.dtype == torch.int32 and got.shape == (3, M)
    assert torch.equal(got, P.furthest_point_sample(x, M))
    if P.ref_available():
        assert torch.equal(got, P.ref_furthest_point_sample(x.to(DEV), M).cpu())


def test_fps_many_small_objects_warp_path():
    from pcreid_b200.ops import furthest_point_sample
    x = O.synth_objects(700, 256, 5, dup=True)
    assert torch.equal(furthest_point_sample(x.to(DEV), 64).cpu(), P.furthest_point_sample(x, 64))


@pytest.mark.parametrize("B,N,M", [(320, 1024, 96), (300, 700, 50), (5, 3000, 40), (3, 8192, 24), (2, 9000, 12)])
def test_fps_rank_kernel_shapes(B, N, M):
    """the shared-memory rank-order FPS kernel: a warp per object with 32 slots per lane (B >= 296, N <= 1024), slot counts that
    are not a power of two (N = 3000: 3 rows of 1024 slots), its largest shape (8192 slots) and the first shape beyond it
    (register kernel); clouds with repeated points so that the tie priority decides"""
    from pcreid_b200.ops import furthest_point_sample
    x = O.synth_objects(B, N, 11, dup=True)
    got = furthest_point_sample(x.to(DEV), M).cpu()
    assert torch.equal(got, P.furthest_point_sample(x, M))
    if P.ref_available() and B <= 8:
        assert torch.equal(got, P.ref_furthest_point_sample(x.to(DEV), M).cpu())


@pytest.mark.parametrize("N", [256, 1000, 3000])
def test_fps_temp_written_back(N):
    """the op's `temp` argument is in/out (furthest_point_sample_cuda.cu:44-70): it ends as the running minimum distance of
    every point to the sample set -- compared with the C restatement's buffer, and a second call that starts from it"""
    import ctypes
    import numpy as np
    from pcreid_b200.ops._common import OPS
    x = O.synth_objects(3, N, 4, dup=True)
    M = 20
    temp = torch.full((3, N), 1e10, device=DEV)
    idx = torch.empty(3, M, dtype=torch.int32, device=DEV)
    OPS.fps(3, N, M, x.to(DEV), temp, idx)
    xn = np.ascontiguousarray(x.numpy())
    tn = np.full((3, N), 1e10, np.float32)
    inn = np.zeros((3, M), np.int32)
    fp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    P._cpu().oracle_fps(3, N, M, fp(xn), fp(tn), fp(inn))
    assert torch.equal(idx.cpu(), torch.from_numpy(inn))
    assert torch.equal(temp.cpu(), torch.from_numpy(tn))
    OPS.fps(3, N, M, x.to(DEV), temp, idx)                # warm start from the buffer
    P._cpu().oracle_fps(3, N, M, fp(xn), fp(tn), fp(inn))
    assert torch.equal(idx.cpu(), torch.from_numpy(inn)) and torch.equal(temp.cpu(), torch.from_numpy(tn))


@pytest.mark.parametrize("N,M", [(128, 32), (100, 100)])
def test_fps_with_dist_bit_exact(N, M):
    from pcreid_b200.ops import furthest_point_sample_with_dist
    x = O.synth_objects(2, N, 2, dup=True)
    d = ((x[:, :, None, :] - x[:, None, :, :]) ** 2).sum(-1).contiguous()
    got = furthest_point_sample_with_dist(d.to(DEV), M).cpu()
    assert torch.equal(got, P.furthest_point_sample_with_dist(d, M))
    if P.ref_available():
        assert torch.equal(got, P.ref_furthest_point_sample_with_dist(d.to(DEV), M).cpu())


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N,S,k", [(256, 256, 32), (256, 128, 48), (160, 80, 48), (1024, 64, 32), (12, 12, 16), (3000, 40, 100)])
def test_knn_op_bit_exact_including_heap_ties(kind, N, S, k):
    from pcreid_b200.ops import knn
    x = clouds(2, N, 3, kind)
    c = x[:, :S].contiguous()
    got = knn(k, x.to(DEV), c.to(DEV), False).cpu()
    assert got.dtype == torch.int32 and got.shape == (2, k, S)
    assert torch.equal(got, P.knn(k, x, c))
    if P.ref_available():
        assert torch.equal(got, P.ref_knn(k, x.to(DEV), c.to(DEV)).cpu())


def test_knn_transposed_and_default_center():
    from pcreid_b200.ops import knn
    x = O.synth_objects(2, 64, 9)
    a = knn(8, x.to(DEV)).cpu()
    b = knn(8, x.permute(0, 2, 1).contiguous().to(DEV), None, True).cpu()
    assert torch.equal(a, P.knn(8, x)) and torch.equal(a, b)
    with pytest.raises(AssertionError):
        knn(101, x.to(DEV))


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N,S,k,rmin,rmax", [(256, 64, 16, 0.0, 0.8), (300, 33, 32, 0.3, 1.5), (64, 64, 64, 0.0, 100.0)])
def test_ball_query_bit_exact(kind, N, S, k, rmin, rmax):
    from pcreid_b200.ops import ball_query
    x = clouds(2, N, 4, kind)
    c = (x[:, :S] + (0.0 if kind != "free" else 0.01)).contiguous()
    got = ball_query(rmin, rmax, k, x.to(DEV), c.to(DEV)).cpu()
    assert torch.equal(got, P.ball_query(rmin, rmax, k, x, c))
    if P.ref_available():
        assert torch.equal(got, P.ref_ball_query(rmin, rmax, k, x.to(DEV), c.to(DEV)).cpu())


@pytest.mark.parametrize("C,N,S,k", [(64, 256, 128, 48), (3, 100, 7, 5), (131, 128, 64, 48)])
def test_group_and_gather_exact(C, N, S, k):
    from pcreid_b200.ops import gather_points, grouping_operation
    g = torch.Generator().manual_seed(0)
    f = torch.randn(2, C, N, generator=g)
    idx = torch.randint(0, N, (2, S, k), generator=g, dtype=torch.int32)
    got = grouping_operation(f.to(DEV), idx.to(DEV)).cpu()
    assert torch.equal(got, P.grouping_operation(f, idx))
    i2 = torch.randint(0, N, (2, S), generator=g, dtype=torch.int32)
    got2 = gather_points(f.to(DEV), i2.to(DEV)).cpu()
    assert torch.equal(got2, P.gather_points(f, i2))
    if P.ref_available():
        assert torch.equal(got, P.ref_grouping_operation(f.to(DEV), idx.to(DEV)).cpu())
        assert torch.equal(got2, P.ref_gather_points(f.to(DEV), i2.to(DEV)).cpu())


def test_query_and_group_and_sampler_modules():
    from pcreid_b200.ops import Points_Sampler, QueryAndGroup
    x = O.synth_objects(2, 128, 6)
    f = torch.randn(2, 16, 128, generator=torch.Generator().manual_seed(1))
    sampler = Points_Sampler([32], ["D-FPS"], [-1])
    fi = sampler(x.to(DEV), f.to(DEV))
    assert torch.equal(fi.cpu(), P.furthest_point_sample(x, 32))
    centers = torch.gather(x, 1, fi.cpu().long().unsqueeze(-1).expand(2, 32, 3)).contiguous()
    for max_r in (None, 0.9):
        qg = QueryAndGroup(max_r, 8, use_xyz=True, return_grouped_idx=True)
        nf, idx = qg(x.to(DEV), centers.to(DEV), f.to(DEV))
        ref_idx = P.knn(8, x, centers).transpose(1, 2).contiguous() if max_r is None else P.ball_query(0, max_r, 8, x, centers)
        assert torch.equal(idx.cpu(), ref_idx)
        gx = P.grouping_operation(x.transpose(1, 2).contiguous(), ref_idx) - centers.transpose(1, 2).unsqueeze(-1)
        ref_nf = torch.cat([gx, P.grouping_operation(f, ref_idx)], dim=1)
        assert torch.equal(nf.cpu(), ref_nf)


@pytest.mark.parametrize("kind", ["free", "dup", "same", "u3"])
@pytest.mark.parametrize("N,S,k", [(256, 256, 32), (256, 128, 48), (128, 64, 48), (160, 80, 48), (1024, 512, 48)])
def test_knn_point_torch_path_canonical(kind, N, S, k):
    """torch-path kNN of the backbones: index-exact vs the oracle's canonical (d, idx) order, whose distances are
    torch's own square_distance (bit-exact restatement checked in test_ops_oracle.py)."""
    import pcreid_b200.kernels as K
    x = clouds(3, N, 7, kind)
    q = x[:, :S].contiguous()
    got = K.knn_point(k, x.to(DEV), q.to(DEV)).cpu().long()
    d = P.sqdist_expand(q, x)
    ref = torch.sort(d, dim=-1, stable=True)[1][..., :k]
    assert torch.equal(got, ref)
    if kind == "free":
        assert torch.equal(got.sort(-1)[0], O.knn_point(k, x, q, canonical=False).sort(-1)[0])


@pytest.mark.parametrize("C,N,k", [(3, 256, 20), (64, 256, 20), (128, 160, 20), (64, 1024, 20)])
def test_knn_feature_canonical(C, N, k):
    import pcreid_b200.kernels as K
    x = torch.randn(2, C, N, generator=torch.Generator().manual_seed(C + N))
    x[:, :, 5] = x[:, :, 9]          # exact duplicate columns -> ties
    got = K.knn_feature(x.to(DEV), k).cpu().long()
    ref = torch.sort(P.dgcnn_pd(x), dim=-1, descending=True, stable=True)[1][..., :k]
    assert torch.equal(got, ref)


def test_golden_knn_vectors():
    import numpy as np
    import helpers
    import pcreid_b200.kernels as K
    g = helpers.golden("knn_torch_path")
    x = torch.from_numpy(g["xyz"])
    got = K.knn_point(48, x.to(DEV), x[:, :80].contiguous().to(DEV)).cpu().long()
    assert torch.equal(got.sort(-1)[0], torch.from_numpy(g["idx"]).long().sort(-1)[0])
    xf = torch.from_numpy(g["feat"])
    gotf = K.knn_feature(xf.to(DEV), 20).cpu().long()
    assert torch.equal(gotf.sort(-1)[0], torch.from_numpy(g["idx_feat"]).long().sort(-1)[0])


def test_reference_cu_kernels_were_compared():
    """The bit-exact comparisons with the reference's own .cu kernels in this file and in test_gpu_frontend.py run only where
    oracle/_ref/ was built from the upstream source tree (PCREID_REFERENCE_ROOT, oracle/Makefile).  Without it they drop out of
    the tests above; this test reports that as a skip instead of letting it pass unnoticed."""
    from oracle import frontend_oracle as F
    missing = [name for name, ok in (("libref_ops.so", P.ref_available()), ("libref_pib.so", F.ref_pib_available())) if not ok]
    if missing:
        pytest.skip(f"oracle/_ref/{' and '.join(missing)} absent, comparisons with the reference .cu kernels left out: "
                    "the upstream source tree is needed to build them")
    x = O.synth_objects(2, 256, 0, dup=True)
    assert torch.equal(P.ref_furthest_point_sample(x.to(DEV), 32).cpu(), P.furthest_point_sample(x, 32))


def test_empty_inputs_are_noops():
    from pcreid_b200.ops import furthest_point_sample, knn
    x = torch.zeros(0, 16, 3, device=DEV)
    assert furthest_point_sample(x, 4).shape == (0, 4)
    assert knn(3, x).shape == (0, 3, 16)


def test_large_scene_scale_sortedness_property():
    """full-size property check (no oracle needed): distances ascending, self is nearest, indices in range."""
    from pcreid_b200.ops import knn
    x = O.synth_objects(8, 4096, 12).to(DEV)
    idx, d2 = knn(32, x, x[:, :1024].contiguous(), False, True)
    assert (d2[:, 1:, :] >= d2[:, :-1, :]).all()
    assert (idx[:, 0, :] == torch.arange(1024, device=DEV, dtype=torch.int32)).all()
    assert int(idx.min()) >= 0 and int(idx.max()) < 4096


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("N,M", [(256, 64), (1000, 37), (64, 2500), (5, 2), (33, 1)])
def test_three_nn_bit_exact(kind, N, M):
    """three_nn (SURVEY 8f row 3): indices and squared distances bit-identical to the C restatement of the reference
    kernel and to the reference .cu itself, including exact ties and fewer than three sources."""
    from pcreid_b200.ops import three_nn
    t, s = clouds(2, N, 3, kind), clouds(2, M, 4 if kind != "same" else 3, kind)
    d, idx = three_nn(t.to(DEV), s.to(DEV))
    d2o, io = P.three_nn_dist2(t, s)
    assert idx.dtype == torch.int32 and torch.equal(idx.cpu(), io)
    assert torch.equal(d, torch.sqrt(d2o.to(DEV)))            # same device for the root: torch's CPU / CUDA sqrt differ in the last bit
    if P.ref_available():
        dr, ir = P.ref_three_nn(t.to(DEV), s.to(DEV))
        assert torch.equal(idx, ir) and torch.equal(d, dr)


@pytest.mark.parametrize("C,M,N", [(64, 128, 256), (3, 7, 1000), (130, 64, 33)])
def test_three_interpolate_bit_exact(C, M, N):
    from pcreid_b200.ops import three_interpolate, three_nn
    f = torch.randn(2, C, M, generator=torch.Generator().manual_seed(0))
    t, s = O.synth_objects(2, N, 5), O.synth_objects(2, M, 6)
    d, idx = three_nn(t.to(DEV), s.to(DEV))
    w = 1.0 / (d + 1e-8)
    w = (w / w.sum(2, keepdim=True)).contiguous()             # PointFPModule.forward weights (point_fp_module.py:60-64)
    out = three_interpolate(f.to(DEV), idx, w)
    assert torch.equal(out.cpu(), P.three_interpolate(f, idx.cpu(), w.cpu()))
    if P.ref_available():
        assert torch.equal(out, P.ref_three_interpolate(f.to(DEV), idx, w))


@pytest.mark.parametrize("radius,nsample,dup", [(0.7, 16, False), (2.5, 48, False), (0.05, 8, True), (1e-4, 4, False)])
def test_query_ball_point_torch_path_exact(radius, nsample, dup):
    """SURVEY 8a A6: pointnet2_utils.query_ball_point (use_knn=False): indices exact, expansion-form distance, d <= r^2"""
    import pcreid_b200.kernels as K
    from oracle import reid_oracle as RO
    x = RO.synth_objects(3, 160, 4, dup=dup)
    q = x[:, :80].contiguous()
    got = K.query_ball_point(radius, nsample, x.to(DEV), q.to(DEV)).cpu()
    assert got.dtype == torch.int32 and torch.equal(got.long(), RO.query_ball_point(radius, nsample, x, q))
    far = (q + 100.0).contiguous()                      # no point within the radius: the reference leaves N in every slot
    assert (K.query_ball_point(radius, nsample, x.to(DEV), far.to(DEV)).cpu() == 160).all()


@pytest.mark.parametrize("fast", [False, True])
def test_sa_layer_with_ball_query_grouping(fast):
    from pcreid_b200.models.pointnet2_utils import PointNetSetAbstractionEdgeSA
    from oracle import reid_oracle as RO
    torch.manual_seed(66)
    sa = PointNetSetAbstractionEdgeSA(npoint=None, radius=1.2, nsample=24, mlp=[0, 32, 32, 32], sampling="RANDOM", use_xyz=True,
                                      use_knn=False).eval()
    sd = RO.perturb_norm_state({"sa." + k: v for k, v in sa.state_dict().items()})
    sa.load_state_dict({k[3:]: v for k, v in sd.items()})
    sa = sa.to(DEV)
    sa.tc_mode = fast
    sa.self_attention.tc_mode = fast
    x = RO.synth_objects(2, 128, 3)
    with torch.no_grad():
        nx, nf = sa(x.to(DEV), None, 64)
    ox, of = RO.sa_layer(sd, "sa", x, None, 64, 24, radius=1.2)
    assert torch.equal(nx.cpu(), ox)
    assert (nf.cpu() - of).abs().max() < (2e-2 if fast else 1e-4)


@pytest.mark.parametrize("B,N,M,dup", [(4, 96, 40, False), (4, 96, 40, True), (3, 1000, 128, False), (600, 128, 32, True), (2, 5000, 64, False)])
def test_farthest_point_sample_torch_path_exact(B, N, M, dup):
    """SURVEY 8a A4: pointnet2_utils.farthest_point_sample (sampling='FPS'): given start indices, (dx*dx + dy*dy) + dz*dz distance,
    lowest index among tied maxima -- indices exact against the oracle (itself bit-exact against the reference function)"""
    import pcreid_b200.kernels as K
    from oracle import reid_oracle as RO
    x = RO.synth_objects(B, N, 3, dup=dup)
    start = torch.randint(0, N, (B,), generator=torch.Generator().manual_seed(1))
    got = K.farthest_point_sample(x.to(DEV), M, start=start).cpu()
    assert got.dtype == torch.int32 and torch.equal(got.long(), RO.farthest_point_sample(x, M, start))
    torch.manual_seed(9)                                  # default start: the reference's host-RNG draw
    got = K.farthest_point_sample(x.to(DEV), M).cpu()
    torch.manual_seed(9)
    assert torch.equal(got.long(), RO.farthest_point_sample(x, M))


@pytest.mark.parametrize("fast,use_knn", [(False, True), (False, False), (True, True)])
def test_sa_layer_with_fps_sampling(fast, use_knn):
    from pcreid_b200.models.pointnet2_utils import PointNetSetAbstractionEdgeSA
    from oracle import reid_oracle as RO
    torch.manual_seed(66)
    sa = PointNetSetAbstractionEdgeSA(npoint=None, radius=1.5, nsample=24, mlp=[64, 64, 64, 64], sampling="FPS", use_xyz=True,
                                      use_knn=use_knn).eval()
    sd = RO.perturb_norm_state({"sa." + k: v for k, v in sa.state_dict().items()})
    sa.load_state_dict({k[3:]: v for k, v in sd.items()})
    sa = sa.to(DEV)
    sa.tc_mode = fast
    sa.self_attention.tc_mode = fast
    x, f = RO.synth_objects(2, 128, 3), torch.randn(2, 32, 128)
    torch.manual_seed(5)
    with torch.no_grad():
        nx, nf = sa(x.to(DEV), f.to(DEV), 64)
    torch.manual_seed(5)
    start = torch.randint(0, 128, (2,), dtype=torch.long)
    ox, of = RO.sa_layer(sd, "sa", x, f, 64, 24, radius=None if use_knn else 1.5, fps_start=start)
    assert torch.equal(nx.cpu(), ox)
    assert (nf.cpu() - of).abs().max() < (2e-2 if fast else 1e-4)
