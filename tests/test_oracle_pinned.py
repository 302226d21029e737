"""Pins the oracle (oracle/reid_oracle.py): (1) bit-exact against the unmodified reference modules where
PCREID_REFERENCE_ROOT names the upstream source tree, (2) against the committed golden vectors everywhere."""
import numpy as np
import pytest
import torch

import helpers
from oracle import ref_loader, reid_oracle as O

needs_ref = pytest.mark.skipif(not ref_loader.available(), reason=ref_loader.MISSING)


def _load_ref_sd(mod, prefix, sd):
    mod.load_state_dict({k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)})


@needs_ref
@pytest.mark.parametrize("canonical", [False, True])
def test_pt_backbone_bit_exact_vs_reference(canonical):
    R = ref_loader.load()
    torch.manual_seed(66)
    bb = R.Pointnet_Backbone(input_channels=0, use_xyz=True, conv_out=64).eval()
    sd = O.perturb_norm_state({"backbone." + k: v for k, v in bb.state_dict().items()})
    _load_ref_sd(bb, "backbone.", sd)
    x = O.synth_objects(3, 160, 0)
    with torch.no_grad():
        _, h_r = bb(x, [160, 80, 40])
        _, h_o = O.pt_backbone(sd, "backbone", x, [160, 80, 40], canonical=canonical)
    assert torch.equal(h_r, h_o)      # tie-free input: canonical (d, idx) order == reference argsort


@needs_ref
@pytest.mark.parametrize("mul,conv_out", [(2, 64), (4, 128)])
def test_pt_backbone_size_variants_bit_exact_vs_reference(mul, conv_out):
    """the 1.5M / 7M configs (reid_pts_point-transformer-{1.5M,7M}_point-cat.py: mul=2 / mul=4)"""
    R = ref_loader.load()
    torch.manual_seed(66)
    bb = R.Pointnet_Backbone(input_channels=0, use_xyz=True, conv_out=conv_out, mul=mul).eval()
    sd = O.perturb_norm_state({"backbone." + k: v for k, v in bb.state_dict().items()})
    _load_ref_sd(bb, "backbone.", sd)
    x = O.synth_objects(2, 128, 0)
    with torch.no_grad():
        _, h_r = bb(x, [128, 64, 32])
        _, h_o = O.pt_backbone(sd, "backbone", x, [128, 64, 32])
    assert torch.equal(h_r, h_o)


@needs_ref
def test_dgcnn_pointnet_heads_bit_exact_vs_reference():
    R = ref_loader.load()
    x = O.synth_objects(2, 128, 1).permute(0, 2, 1).contiguous()
    torch.manual_seed(66)
    dg = R.DGCNN().eval()
    sd = O.perturb_norm_state({"backbone." + k: v for k, v in dg.state_dict().items()})
    _load_ref_sd(dg, "backbone.", sd)
    pn = R.PointNet(k=40, normal_channel=False).eval()
    sdp = O.perturb_norm_state({"backbone." + k: v for k, v in pn.state_dict().items()})
    _load_ref_sd(pn, "backbone.", sdp)
    ca = R.corss_attention(d_model=64, nhead=2).eval()
    sdc = O.perturb_norm_state({"cross_stage1." + k: v for k, v in ca.state_dict().items()})
    _load_ref_sd(ca, "cross_stage1.", sdc)
    lr = R.LinearRes(1024, 512, norm='GN', ng=64).eval()
    sdl = O.perturb_norm_state({"d." + k: v for k, v in lr.state_dict().items()})
    _load_ref_sd(lr, "d.", sdl)
    s, t = torch.randn(3, 64, 128), torch.randn(3, 64, 96)
    sx, tx = torch.randn(3, 128, 3), torch.randn(3, 96, 3)
    r = torch.randn(10, 1024)
    with torch.no_grad():
        assert torch.equal(dg(x, None)[1], O.dgcnn_backbone(sd, "backbone", x, 20, canonical=True)[1])
        assert torch.equal(pn(x, None)[1], O.pointnet_backbone(sdp, "backbone", x)[1])
        assert torch.equal(ca(s, sx, t, tx), O.cross_attention(sdc, "cross_stage1", s, sx, t, tx))
        assert torch.equal(lr(r), O.linear_res(sdl, "d", r, 64))


@needs_ref
@pytest.mark.parametrize("canonical", [True, False])
def test_local_self_attention_bit_exact_vs_reference(canonical):
    """the 'xcorr' match type's local stage (attention.py:221-296) against the unmodified reference module"""
    R = ref_loader.load()
    torch.manual_seed(66)
    ls = R.local_self_attention(d_model=64, nhead=2, attention='linear', knum=48, pos_size=64).eval()
    sd = O.perturb_norm_state({"local_stage1." + k: v for k, v in ls.state_dict().items()})
    _load_ref_sd(ls, "local_stage1.", sd)
    f, x = torch.randn(3, 64, 128), O.synth_objects(3, 128, 5)
    with torch.no_grad():
        ref = ls(f, x)
        got = O.local_self_attention(sd, "local_stage1", f, x, 48, canonical=canonical)
    if canonical:
        assert (ref - got).abs().max() < 1e-6       # tie order of topk is the only freedom (none on random input)
    else:
        assert torch.equal(ref, got)


@needs_ref
def test_product_modules_reproduce_reference_init_and_keys():
    """seed-66 default init of the product's modules == the reference's, key for key (so goldens travel)."""
    R = ref_loader.load()
    from pcreid_b200.models import DGCNN, LinearRes, PointNet, Pointnet_Backbone, corss_attention
    for mine, ref in ((lambda: Pointnet_Backbone(input_channels=0, use_xyz=True, conv_out=64),
                       lambda: R.Pointnet_Backbone(input_channels=0, use_xyz=True, conv_out=64)),
                      (DGCNN, R.DGCNN), (lambda: PointNet(k=40, normal_channel=False), lambda: R.PointNet(k=40, normal_channel=False)),
                      (lambda: corss_attention(64, 2), lambda: R.corss_attention(64, 2)),
                      (lambda: LinearRes(1024, 512, ng=64), lambda: R.LinearRes(1024, 512, ng=64))):
        torch.manual_seed(66)
        a = mine().state_dict()
        torch.manual_seed(66)
        b = ref().state_dict()
        assert list(a.keys()) == list(b.keys())
        assert all(torch.equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("name,kind,tol", [("reid_pt", "pt", 2e-5), ("reid_pt256", "pt", 2e-5), ("reid_dgcnn", "dgcnn", 2e-5),
                                           ("reid_pointnet", "pointnet", 2e-5), ("reid_xcorr", "xcorr", 2e-5),
                                           ("reid_xcorr-baseline", "xcorr-baseline", 2e-5)])
def test_oracle_matches_golden(name, kind, tol):
    """Goldens were produced by the reference modules (oracle/make_golden.py); tolerance covers BLAS/CPU differences
    between the generating machine and this one (bit-exact on the generating machine)."""
    g = helpers.golden(name)
    _, orc = helpers.build_pair(kind, tuple(int(v) for v in g["backbone_list"]))
    assert abs(helpers.weight_checksum(orc.sd) - float(g["weight_checksum"])) < 1e-6 * float(g["weight_checksum"])
    t, d = torch.from_numpy(g["tracks"]), torch.from_numpy(g["dets"])
    xt, ht = orc.encode(t)
    xd, hd = orc.encode(d)
    assert (ht - torch.from_numpy(g["h_t"])).abs().max() < tol
    assert (hd - torch.from_numpy(g["h_d"])).abs().max() < tol
    L = orc.match_all_pairs(ht, xt, hd, xd)
    assert (L - torch.from_numpy(g["logits"])).abs().max() < tol


def test_knn_golden_and_canonical_order():
    g = helpers.golden("knn_torch_path")
    """golden = the reference's own knn_point (unstable argsort) / dgcnn knn (topk) output.  The canonical (d, idx)
    order must select the same neighbour set with the same ordered distance list; positions may differ only inside
    exact-distance ties (continuous random input still has a few: 1 tied pair in 11520 entries here)."""
    x = torch.from_numpy(g["xyz"])
    ref, can = torch.from_numpy(g["idx"]).long(), O.knn_point(48, x, x[:, :80], canonical=True)
    d = O.square_distance(x[:, :80], x)
    assert torch.equal(torch.gather(d, 2, ref), torch.gather(d, 2, can))
    assert torch.equal(ref.sort(-1)[0], can.sort(-1)[0])
    assert (ref != can).float().mean() < 1e-3
    xf = torch.from_numpy(g["feat"])
    reff, canf = torch.from_numpy(g["idx_feat"]).long(), O.dgcnn_knn(xf, 20, canonical=True)
    pd = O.dgcnn_pairwise(xf)
    assert torch.equal(torch.gather(pd, 2, reff), torch.gather(pd, 2, canf))
    assert torch.equal(reff.sort(-1)[0], canf.sort(-1)[0])


def test_class_gate_matches_tracker_semantics():
    lt = torch.tensor([0, 1, 1, 9, 3]); nt = torch.tensor([5, 1, 7, 9, 2])
    ld = torch.tensor([1, 1, 3, 9]); nd = torch.tensor([4, 0, 2, 8])
    m = O.class_gated_pairs(lt, nt, ld, nd)
    assert m.tolist() == [[False] * 4, [False] * 4, [True, False, False, False], [False] * 4, [False, False, True, False]]


@needs_ref
def test_cross_lin_attn_bit_exact_vs_reference():
    """image-token cross block (attention.py:312-372) against the unmodified reference module, 198 tokens"""
    R = ref_loader.load()
    torch.manual_seed(66)
    ca = R.cross_lin_attn(d_model=64, nhead=2).eval()
    sd = O.perturb_norm_state({"cross_stage1." + k: v for k, v in ca.state_dict().items()})
    _load_ref_sd(ca, "cross_stage1.", sd)
    a, b = O.synth_tokens(3, 64, 198, 0), O.synth_tokens(3, 64, 77, 1)
    with torch.no_grad():
        assert torch.equal(ca(a, b), O.cross_lin_attention(sd, "cross_stage1", a, b))


@needs_ref
def test_image_modules_reproduce_reference_init_and_keys():
    from pcreid_b200.models import cross_lin_attn
    R = ref_loader.load()
    torch.manual_seed(66)
    a = cross_lin_attn(64, 2).state_dict()
    torch.manual_seed(66)
    b = R.cross_lin_attn(64, 2).state_dict()
    assert list(a.keys()) == list(b.keys()) and all(torch.equal(a[k], b[k]) for k in a)


def test_image_oracle_matches_golden():
    """golden = reference cross_lin_attn / LinearRes / nn.Linear modules assembled as ImageReIDNet does (oracle/make_golden.py)"""
    g = helpers.golden("reid_image_tokens")
    _, orc = helpers.build_image_pair()
    assert abs(helpers.weight_checksum(orc.sd) - float(g["weight_checksum"])) < 1e-6 * float(g["weight_checksum"])
    assert (orc.downsample_tokens(torch.from_numpy(g["raw"])) - torch.from_numpy(g["h_raw"])).abs().max() < 2e-5
    L = orc.match_all_pairs(torch.from_numpy(g["h_t"]), torch.from_numpy(g["h_d"]))
    assert (L - torch.from_numpy(g["logits"])).abs().max() < 2e-5


@needs_ref
@pytest.mark.parametrize("radius,nsample", [(0.7, 16), (2.5, 48), (0.05, 8)])
def test_query_ball_point_bit_exact_vs_reference(radius, nsample):
    """SURVEY 8a A6: the torch-path ball query (pointnet2_utils.py:218-240), reachable with use_knn=False"""
    R = ref_loader.load()
    x = O.synth_objects(3, 160, 4, dup=(nsample == 8))
    ref = R.pointnet2_utils.query_ball_point(radius, nsample, x, x[:, :80].contiguous())
    assert torch.equal(ref, O.query_ball_point(radius, nsample, x, x[:, :80].contiguous()))


@needs_ref
def test_sa_layer_with_ball_query_bit_exact_vs_reference():
    R = ref_loader.load()
    torch.manual_seed(66)
    sa = R.pointnet2_utils.PointNetSetAbstractionEdgeSA(npoint=None, radius=1.2, nsample=24, mlp=[0, 32, 32, 32], sampling="RANDOM",
                                                        use_xyz=True, use_knn=False).eval()
    sd = O.perturb_norm_state({"sa." + k: v for k, v in sa.state_dict().items()})
    _load_ref_sd(sa, "sa.", sd)
    x = O.synth_objects(2, 128, 3)
    with torch.no_grad():
        rx, rf = sa(x, None, 64)
    ox, of = O.sa_layer(sd, "sa", x, None, 64, 24, radius=1.2)
    assert torch.equal(rx, ox) and torch.equal(rf, of)


@needs_ref
@pytest.mark.parametrize("dup", [False, True])
def test_farthest_point_sample_bit_exact_vs_reference(dup):
    """SURVEY 8a A4: the torch-path FPS (pointnet2_utils.py:116-137) incl. its host-RNG start and torch.max tie behaviour"""
    R = ref_loader.load()
    x = O.synth_objects(4, 96, 3, dup=dup)
    torch.manual_seed(11)
    ref = R.pointnet2_utils.farthest_point_sample(x, 40)
    torch.manual_seed(11)
    assert torch.equal(ref, O.farthest_point_sample(x, 40))
    torch.manual_seed(11)
    start = torch.randint(0, 96, (4,), dtype=torch.long)
    assert torch.equal(ref, O.farthest_point_sample(x, 40, start))


@needs_ref
@pytest.mark.parametrize("use_knn", [True, False])
def test_sa_layer_with_fps_sampling_bit_exact_vs_reference(use_knn):
    R = ref_loader.load()
    torch.manual_seed(66)
    sa = R.pointnet2_utils.PointNetSetAbstractionEdgeSA(npoint=None, radius=1.5, nsample=24, mlp=[64, 64, 64, 64], sampling="FPS",
                                                        use_xyz=True, use_knn=use_knn).eval()
    sd = O.perturb_norm_state({"sa." + k: v for k, v in sa.state_dict().items()})
    _load_ref_sd(sa, "sa.", sd)
    x, f = O.synth_objects(2, 128, 3), torch.randn(2, 32, 128)
    torch.manual_seed(5)
    with torch.no_grad():
        rx, rf = sa(x, f, 64)
    torch.manual_seed(5)
    start = torch.randint(0, 128, (2,), dtype=torch.long)
    ox, of = O.sa_layer(sd, "sa", x, f, 64, 24, radius=None if use_knn else 1.5, fps_start=start)
    assert torch.equal(rx, ox) and torch.equal(rf, of)
