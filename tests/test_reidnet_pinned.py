"""Pins the oracle AND the product's reference-facing API to the reference's OWN ReIDNet / ImageReIDNet classes:
mmdet3d/models/ReIDNet.py is imported unmodified by path (oracle/ref_loader.load_reidnet; stand-ins only for the mmcv registry,
mmdet's BaseDetector base class and pytorch3d's training-only chamfer loss) and run on CPU under the shipped configs
(configs_reid/_base_/reidentifiers/*.py + the losses_to_use / alpha of configs_reid/reid_nuscenes_pts/*.py).

  * oracle.ReIDOracle / ImageReIDOracle == the real classes, bit for bit (siamese_forward, xcorr_eff, get_pooled_feats,
    match_forward_inference, forward_test);
  * the product's modules (with the kernel *specification* emulation of tests/fake_kernels.py on CPU) return the same result
    dict as the real forward_test, key for key, and load the real class's state_dict with strict=True.
Runs where PCREID_REFERENCE_ROOT names the upstream source tree."""
import copy

import pytest
import torch

import fake_kernels
import helpers
from oracle import ref_loader, reid_oracle as O

pytestmark = pytest.mark.skipif(not ref_loader.available(), reason=ref_loader.MISSING)

SHIPPED = dict(losses_to_use=dict(kl=False, match=True, cls=False, shape=False, fp=False, triplet=False),
               alpha=dict(kl=1, match=1, cls=1, shape=1, fp=1, vis=1, triplet=1), triplet_loss=dict(margin=10, p=2),
               triplet_sample_num=128)


@pytest.fixture(scope="module")
def R():
    return ref_loader.load_reidnet()


@pytest.fixture()
def fake(monkeypatch):
    fake_kernels.install(monkeypatch)


def _build_ref(R, kind, blist=(128, 64, 32)):
    cfg = copy.deepcopy(helpers.model_cfg(kind, blist))
    cfg.pop("type")
    cfg.update(copy.deepcopy(SHIPPED))
    torch.manual_seed(66)
    net = R.ReIDNet(**cfg).eval()
    sd = O.perturb_norm_state(net.state_dict())
    net.load_state_dict(sd)
    return net, sd


def _batch(n, N, seed):
    s1, s2 = O.synth_objects(n, N, seed), O.synth_objects(n, N, seed + 1)
    one = lambda v: [torch.tensor([x]) for x in v]
    ids1, ids2 = list(range(n)), [i if i % 2 == 0 else 100 + i for i in range(n)]
    return dict(sparse_1=list(s1), sparse_2=list(s2), dense_1=list(s1), dense_2=list(s2), label_1=one([1, 2, 12][:n]),
                label_2=one([1, 2, 3][:n]), id_1=one(ids1), id_2=one(ids2), size_1=one([9] * n), size_2=one([7] * n),
                vis_1=one([1] * n), vis_2=one([2] * n)), s1, s2


@pytest.mark.parametrize("kind", ["pt", "concat", "dgcnn", "pointnet", "xcorr", "xcorr-baseline", "pt15m", "pt7m"])
def test_oracle_equals_the_real_reidnet_class(R, kind):
    net, sd = _build_ref(R, kind)
    # canonical=False: the oracle uses the reference's own argsort / topk calls, so even the order of the neighbours (and with it
    # the summation order inside local_self_attention) is the reference's
    orc = O.ReIDOracle(sd, backbone_list=(128, 64, 32), canonical=False, **helpers.ORACLE_KW[kind])
    data, s1, s2 = _batch(3, 128, 2)
    with torch.no_grad():
        x1, x2, h1, h2 = net.siamese_forward(s1, s2)
        res = net(return_loss=False, **data)[0]
        if kind == "xcorr-baseline":     # only match_forward (the forward_test path, ReIDNet.py:398-406) knows this type;
            with pytest.raises(NotImplementedError):                  # match_forward_inference (444-460) rejects it
                net.match_forward_inference(h1, h2, x1, x2)
            lg = res['val_match_preds']
        else:
            lg = net.match_forward_inference(h1, h2, x1, x2)
    o = orc.siamese_forward(s1, s2)
    assert torch.equal(h1, o[2]) and torch.equal(h2, o[3]) and torch.equal(x1, o[0])
    assert torch.equal(lg, orc.match_forward_inference(o[2], o[3], o[0], o[1]))
    assert torch.equal(res['val_match_preds'], lg) and res['val_match_gt'].tolist() == [1., 0., 1.]
    if kind == "pt":
        out, o1, o2 = net.xcorr_eff(h1, x1, h2, x2)
        oo = O.xcorr_eff(sd, o[2], o[0], o[3], o[1], "point-cat")
        assert torch.equal(out, oo[0]) and torch.equal(net.get_pooled_feats(out), O.pooled_feats(oo[0], "both"))
        # the all-pairs driver of the oracle == the real class scored pair by pair
        L = orc.match_all_pairs(o[2], o[0], o[3], o[1])
        with torch.no_grad():
            for i in range(3):
                for j in range(3):       # batch of one pair vs batch of nine: BLAS blocking differs in the last bit
                    one = net.match_forward_inference(h1[i:i + 1], h2[j:j + 1], x1[i:i + 1], x2[j:j + 1])[0]
                    assert abs(float(L[i, j] - one)) < 1e-6


@pytest.mark.parametrize("kind,kl", [("pt", False), ("concat", False), ("dgcnn", False), ("xcorr-baseline", False), ("pt", True)])
def test_product_forward_test_equals_the_real_class(R, fake, kind, kl, monkeypatch):
    from pcreid_b200.models import build_model
    shipped = copy.deepcopy(SHIPPED)
    shipped["losses_to_use"]["kl"] = kl          # kl=True: the validation-only KL term over the embeddings (ReIDNet.py:467-482)
    monkeypatch.setitem(globals(), "SHIPPED", shipped)
    net, sd = _build_ref(R, kind)
    cfg = copy.deepcopy(helpers.model_cfg(kind, (128, 64, 32)))
    cfg.update(copy.deepcopy(shipped))
    mine = build_model(cfg).eval()
    mine.load_state_dict(net.state_dict(), strict=True)              # the real class's checkpoint loads unchanged
    assert list(mine.state_dict().keys()) == list(net.state_dict().keys())
    data, _, _ = _batch(3, 128, 4)
    with torch.no_grad():
        ref = net(return_loss=False, **copy.deepcopy(data))[0]
        got = mine(return_loss=False, **copy.deepcopy(data))[0]
    assert set(got.keys()) == set(ref.keys())
    for k, v in ref.items():
        if v is None:
            assert got[k] is None, k
        elif v.dtype.is_floating_point:
            assert (got[k].float().cpu() - v.float()).abs().max() < 2e-5, k
        else:
            assert torch.equal(got[k].cpu(), v), k


def test_module_factory_names_match(R):
    from pcreid_b200.models import module_obj
    assert set(R.module_obj) - set(module_obj) <= {"PostRes"}         # the only reference factory name not built here
    assert R.build_module(None) is None and R.build_module({}) is None


def test_image_oracle_and_product_equal_the_real_image_class(R, fake, monkeypatch):
    """ImageReIDNet with its HuggingFace backbone replaced by a toy token producer (get_image_model needs the hub)."""
    from pcreid_b200.models import build_model

    class Out:
        def __init__(self, t):
            self.hidden_states = (None, t)

    class Toy(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.proj = torch.nn.Linear(192, 198 * 192)

        def forward(self, pixel_values):
            return Out(self.proj(pixel_values.reshape(pixel_values.shape[0], -1)).reshape(-1, 198, 192))

    torch.manual_seed(1)
    toy = Toy().eval()
    monkeypatch.setattr(R.ReIDNet_module, "get_image_model", lambda name: (None, toy))
    cfg = copy.deepcopy(helpers.image_cfg())
    cfg.pop("type")
    cfg["alpha"] = dict(kl=1, match=1, cls=1, shape=1, fp=1, triplet=1, vis=1)
    torch.manual_seed(66)
    net = R.ImageReIDNet(**copy.deepcopy(cfg)).eval()
    sd = O.perturb_norm_state({k: v for k, v in net.state_dict().items() if not k.startswith("backbone.")})
    net.load_state_dict(sd, strict=False)
    orc = O.ImageReIDOracle(sd, downsample_dim=64, downsample_ng=(32, 16), head_ng=16)
    h_t, h_d = O.synth_tokens(3, 64, 198, 1), O.synth_tokens(3, 64, 198, 2)
    with torch.no_grad():
        assert torch.equal(net.xcorr_eff(h_t, h_d), O.image_xcorr_eff(sd, h_t, h_d))
        assert torch.equal(net.match_forward_inference(h_t, h_d), orc.match_forward_inference(h_t, h_d))
    # forward_test of the real class vs the product (same toy backbone attached)
    mine = build_model(dict(helpers.image_cfg(), alpha=cfg["alpha"])).eval()
    mine.load_state_dict(sd, strict=True)
    mine.set_backbone(toy, name="deit-tiny")
    s1, s2 = torch.randn(3, 3, 8, 8), torch.randn(3, 3, 8, 8)
    one = lambda v: [torch.tensor([x]) for x in v]
    data = dict(sparse_1=list(s1), sparse_2=list(s2), label_1=one([1, 2, 12]), label_2=one([1, 2, 3]), vis_1=one([0, 1, -1]),
                vis_2=one([2, 3, 1]), id_1=one([5, 6, 7]), id_2=one([5, 9, 7]), size_1=one([4, 4, 4]), size_2=one([4, 4, 4]))
    with torch.no_grad():
        ref = net(return_loss=False, **copy.deepcopy(data))[0]
        got = mine(return_loss=False, **copy.deepcopy(data))[0]
    for k in ("val_match_preds", "val_match_gt", "val_cls_preds", "val_fp_preds", "val_vis_preds", "val_cls_gt", "val_vis_gt",
              "val_fp_gt", "match_classes", "num_points", "val_vis_gt_all", "val_match_loss"):
        assert (got[k].float() - ref[k].float()).abs().max() < 2e-5, k
    assert set(ref.keys()) == set(got.keys())


@pytest.mark.parametrize("name,kind", [("reid_pt", "pt"), ("reid_pt256", "pt"), ("reid_dgcnn", "dgcnn"), ("reid_pointnet", "pointnet"),
                                       ("reid_xcorr", "xcorr"), ("reid_xcorr-baseline", "xcorr-baseline")])
def test_committed_goldens_are_outputs_of_the_real_class(R, name, kind):
    """tests/golden/*.npz (what pins parity on the GPU box, where the reference tree is absent) == the real ReIDNet class run
    here on the stored inputs (1e-5: the batch composition differs from the generating run)."""
    g = helpers.golden(name)
    net, sd = _build_ref(R, kind, tuple(int(v) for v in g["backbone_list"]))
    assert abs(helpers.weight_checksum(sd) - float(g["weight_checksum"])) < 1e-6 * float(g["weight_checksum"])
    t, d = torch.from_numpy(g["tracks"]), torch.from_numpy(g["dets"])
    T, D = t.shape[0], d.shape[0]
    n = max(T, D)                                   # siamese_forward wants equally many objects on both sides: pad by repetition
    tt = torch.cat([t, t[:1].expand(n - T, -1, -1)]) if T < n else t
    dd = torch.cat([d, d[:1].expand(n - D, -1, -1)]) if D < n else d
    with torch.no_grad():
        x1, x2, h1, h2 = net.siamese_forward(tt, dd)
        ht, hd, xt, xd = h1[:T], h2[:D], x1[:T], x2[:D]
        pairs = torch.cartesian_prod(torch.arange(T), torch.arange(D))
        a, b = pairs[:, 0], pairs[:, 1]
        if kind == "xcorr-baseline":
            lg = net.match_head(net.get_pooled_feats(net.xcorr_baseline(ht[a], xt[a], hd[b], xd[b]))).squeeze(1)
        else:
            lg = net.match_forward_inference(ht[a], hd[b], xt[a], xd[b])
    # bit-exact when the batch composition equals the generating run; BLAS blocking moves the last bit otherwise
    assert (ht - torch.from_numpy(g["h_t"])).abs().max() < 1e-5 and (hd - torch.from_numpy(g["h_d"])).abs().max() < 1e-5
    assert (lg.reshape(T, D) - torch.from_numpy(g["logits"])).abs().max() < 1e-5
