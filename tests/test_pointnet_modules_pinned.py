"""Pins oracle/pointnet_modules_oracle.py (the CPU restatement the GPU tests of the mmdet3d PointNet++ module family compare
against) to the reference's OWN module code: ops/pointnet_modules/{point_sa_module,point_fp_module,builder}.py,
ops/group_points/group_points.py and ops/furthest_point_sample/{points_sampler,utils}.py are imported unmodified by path
(oracle/ref_loader.load_pointnet_modules) and run on CPU, with the compiled CUDA ops replaced by the op oracle (itself pinned
to the reference .cu files on the GPU box) and mmcv's ConvModule by a torch stand-in.  Runs where PCREID_REFERENCE_ROOT names the upstream source tree."""
import pytest
import torch

from oracle import pointnet_modules_oracle as PO
from oracle import ref_loader, reid_oracle as O

pytestmark = pytest.mark.skipif(not ref_loader.pointnet_modules_available(), reason=ref_loader.MISSING)


def _randomise_bn(m, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.weight.copy_(1 + 0.3 * torch.randn(mod.weight.shape, generator=g))
                mod.bias.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_mean.copy_(0.2 * torch.randn(mod.bias.shape, generator=g))
                mod.running_var.copy_(0.5 + torch.rand(mod.bias.shape, generator=g))
    return m


@pytest.fixture(scope="module")
def R():
    return ref_loader.load_pointnet_modules()


@pytest.mark.parametrize("normalize,dilated,use_feat,pool,fps", [
    (False, False, True, "max", ["D-FPS"]), (True, True, True, "max", ["D-FPS"]), (False, False, False, "max", ["D-FPS"]),
    (False, False, True, "avg", ["D-FPS"]), (False, True, True, "avg", ["F-FPS"]), (True, False, True, "max", ["FS"])])
def test_sa_module_msg_glue_bit_exact_vs_reference(R, normalize, dilated, use_feat, pool, fps):
    torch.manual_seed(3)
    cin = 6 if use_feat else 0
    npt = 24 if fps == ["FS"] else 48
    m = _randomise_bn(R.PointSAModuleMSG(num_point=npt, radii=[0.6, 1.2], sample_nums=[16, 32], mlp_channels=[[cin, 16, 32], [cin, 32, 32, 32]],
                                         normalize_xyz=normalize, dilated_group=dilated, pool_mod=pool, fps_mod=fps,
                                         fps_sample_range_list=[-1]), 1).eval()
    xyz = O.synth_objects(3, 200, 7)
    feat = torch.randn(3, cin, 200) if use_feat else None
    with torch.no_grad():
        nx, nf, idx = m(xyz, feat)
    ox, of, oidx = PO.sa_module_msg(m.state_dict(), npt, [0.6, 1.2], [16, 32], xyz, feat, normalize_xyz=normalize, dilated_group=dilated,
                                    pool_mod=pool, fps_mod=fps, sqdist=R.calc_square_dist)
    assert torch.equal(idx.long(), oidx.long()) and torch.equal(nx, ox) and torch.equal(nf, of)


def test_sa_module_builder_and_group_all_vs_reference(R):
    torch.manual_seed(4)
    m = _randomise_bn(R.build_sa_module(dict(type="PointSAModule", mlp_channels=[29, 32, 32, 32], num_point=40, radius=0.9,
                                             num_sample=24)), 3).eval()
    assert isinstance(m, R.PointSAModule)
    xyz, feat = O.synth_objects(2, 150, 8), torch.randn(2, 29, 150)
    with torch.no_grad():
        nx, nf, idx = m(xyz, feat)
    ox, of, oidx = PO.sa_module_msg(m.state_dict(), 40, [0.9], [24], xyz, feat)
    assert torch.equal(idx.long(), oidx.long()) and torch.equal(nx, ox) and torch.equal(nf, of)
    # num_point=None (GroupAll): this reference version rejects it in BasePointSAModule.__init__ (point_sa_module.py:67-72);
    # the product and the oracle follow upstream mmdet3d (one group holding every point) -- a superset, not a divergence
    with pytest.raises(NotImplementedError):
        R.PointSAModule(mlp_channels=[29, 64, 128])
    g = R.GroupAll(use_xyz=True)                      # the grouper itself is the reference's (group_points.py:132-166)
    got = g(xyz, None, feat)
    assert torch.equal(got, torch.cat([xyz.transpose(1, 2).unsqueeze(2), feat.unsqueeze(2)], dim=1))


@pytest.mark.parametrize("with_target", [True, False])
def test_fp_module_glue_bit_exact_vs_reference(R, with_target):
    torch.manual_seed(5)
    cin = 32 + (16 if with_target else 0)
    m = _randomise_bn(R.PointFPModule(mlp_channels=[cin, 64, 32]), 2).eval()
    target, source = O.synth_objects(2, 120, 1), O.synth_objects(2, 40, 2)
    tf = torch.randn(2, 16, 120) if with_target else None
    sf = torch.randn(2, 32, 40)
    with torch.no_grad():
        ref = m(target, source, tf, sf)
    assert torch.equal(ref, PO.fp_module(m.state_dict(), target, source, tf, sf))


@pytest.mark.parametrize("mods,ranges,npts", [(["F-FPS"], [-1], [32]), (["FS"], [-1], [24]), (["D-FPS", "F-FPS"], [64, -1], [16, 16])])
def test_points_sampler_vs_reference(R, mods, ranges, npts):
    xyz = O.synth_objects(3, 160, 11)
    feat = torch.randn(3, 32, 160, generator=torch.Generator().manual_seed(5))
    ref = R.Points_Sampler(npts, mods, ranges)(xyz, feat)
    assert torch.equal(ref.long(), PO.points_sampler(xyz, feat, npts, mods, ranges, sqdist=R.calc_square_dist).long())
    assert torch.equal(ref.long(), PO.points_sampler(xyz, feat, npts, mods, ranges).long())       # kernel-arithmetic distances
    assert torch.equal(R.calc_square_dist(xyz, xyz, norm=False), PO.calc_square_dist_ref(xyz, xyz, norm=False))


@pytest.mark.parametrize("max_r,normalize,uniform,use_xyz,use_feat", [
    (None, False, False, True, True), (0.9, True, False, True, True), (0.9, False, True, True, True), (0.7, False, True, True, False),
    (0.9, False, False, False, True)])
def test_query_and_group_oracle_vs_reference_class(R, max_r, normalize, uniform, use_xyz, use_feat):
    """oracle.query_and_group_full (what the GPU QueryAndGroup is compared with) equals the reference's own QueryAndGroup,
    including the uniform_sample branch under the same host-generator seed."""
    x = O.synth_objects(2, 96, 6)
    f = torch.randn(2, 5, 96, generator=torch.Generator().manual_seed(1)) if use_feat else None
    centers = x[:, :12].contiguous()
    qg = R.QueryAndGroup(max_r, 8, use_xyz=use_xyz, normalize_xyz=normalize, uniform_sample=uniform, return_grouped_xyz=True,
                         return_unique_cnt=uniform, return_grouped_idx=True)
    torch.manual_seed(11)
    ref = qg(x, centers, f)
    torch.manual_seed(11)
    nf, gx, cnt, idx = PO.query_and_group_full(x, centers, f, max_r, 8, use_xyz=use_xyz, normalize_xyz=normalize, uniform_sample=uniform)
    assert torch.equal(ref[0], nf) and torch.equal(ref[1], gx) and torch.equal(ref[-1], idx)
    if uniform:
        assert torch.equal(ref[2], cnt)


def test_product_modules_have_the_reference_state_dict_keys(R):
    from pcreid_b200.ops import PointFPModule, PointSAModuleMSG
    kw = dict(num_point=48, radii=[0.6, 1.2], sample_nums=[16, 32], mlp_channels=[[6, 16, 32], [6, 32, 32, 32]])
    torch.manual_seed(0)
    a = PointSAModuleMSG(**{k: ([list(c) for c in v] if k == "mlp_channels" else v) for k, v in kw.items()}).state_dict()
    torch.manual_seed(0)
    b = R.PointSAModuleMSG(**{k: ([list(c) for c in v] if k == "mlp_channels" else v) for k, v in kw.items()}).state_dict()
    assert list(a.keys()) == list(b.keys()) and all(a[k].shape == b[k].shape for k in a)
    a, b = PointFPModule(mlp_channels=[48, 64, 32]).state_dict(), R.PointFPModule(mlp_channels=[48, 64, 32]).state_dict()
    assert list(a.keys()) == list(b.keys()) and all(a[k].shape == b[k].shape for k in a)
