"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the UNMODIFIED reference modules
(imported by path from $PCREID_REFERENCE_ROOT through oracle/ref_loader.py) on seeded synthetic inputs.

    python oracle/make_golden.py          # needs PCREID_REFERENCE_ROOT=<upstream source tree>

The reference ships no golden vectors (SURVEY.md section 4); these fixtures are what pins the oracle and
the CUDA path on machines where the reference tree is absent (the GPU box).  Weights are the reference
modules' default init under torch.manual_seed(66) (reference `seed`, reidentification_runtime.py:16)
followed by oracle.reid_oracle.perturb_norm_state (deterministic de-trivialisation of norm statistics);
the product's modules reproduce them bit-for-bit from the same seed (asserted by a checksum).
The ReIDNet glue (ReIDNet.py:311-332, 231-247, 526-534, 444-462) is restated below on top of the reference's own
corss_attention / LinearRes / nn.Linear modules; tests/test_reidnet_pinned.py verifies that the committed vectors are the
outputs of the reference's real ReIDNet class (imported by oracle/ref_loader.load_reidnet) on the stored inputs.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader, reid_oracle as O   # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def checksum(sd):
    return float(sum(v.double().abs().sum() for k, v in sorted(sd.items()) if v.dtype.is_floating_point))


def build_reference(R, kind, local=False):
    """Reference modules in ReIDNet.__init__ construction order (backbone, match_head, downsample, cross_stage1,
    local_stage1, cross_stage2, local_stage2; ReIDNet.py:125-136)."""
    torch.manual_seed(66)
    mods = {}
    if kind == "pt":
        mods["backbone"] = R.Pointnet_Backbone(input_channels=0, use_xyz=True, conv_out=64)
        ng = 8
    elif kind == "dgcnn":
        mods["backbone"] = R.DGCNN(dropout=0.5, emb_dims=1024, k=20, output_channels=40)
        ng = 16
    else:
        mods["backbone"] = R.PointNet(k=40, normal_channel=False)
        ng = 8
    mods["match_head"] = torch.nn.Sequential(R.LinearRes(128, 128, norm='GN', ng=ng), torch.nn.Linear(128, 1))
    if kind != "pt":
        mods["downsample"] = torch.nn.Sequential(R.LinearRes(1024, 512, norm='GN', ng=64), R.LinearRes(512, 128, norm='GN', ng=16),
                                                 torch.nn.Linear(128, 64))
    mods["cross_stage1"] = R.corss_attention(d_model=64, nhead=2, attention='linear')
    if local:   # reid_pts_point-transformer_baseline_orig.py
        mods["local_stage1"] = R.local_self_attention(d_model=64, nhead=2, attention='linear', knum=48, pos_size=64)
    mods["cross_stage2"] = R.corss_attention(d_model=64, nhead=2, attention='linear')
    if local:
        mods["local_stage2"] = R.local_self_attention(d_model=64, nhead=2, attention='linear', knum=48, pos_size=64)
    net = torch.nn.ModuleDict(mods).eval()
    sd = O.perturb_norm_state(net.state_dict())
    net.load_state_dict(sd)
    return net, sd


@torch.no_grad()
def ref_encode(net, kind, pts, blist):
    if kind == "pt":
        return net["backbone"](pts, blist)
    _, h = net["backbone"](pts.permute(0, 2, 1), blist)
    B, C, N = h.shape
    h = net["downsample"](h.permute(0, 2, 1).reshape(-1, C)).reshape(B, N, -1).permute(0, 2, 1)
    return pts, h


@torch.no_grad()
def ref_match(net, h1, h2, xyz1, xyz2):
    a = net["cross_stage1"](h1, xyz1, h2, xyz2)
    b = net["cross_stage1"](h2, xyz2, h1, xyz1)
    o1 = net["cross_stage2"](a, xyz1, b, xyz2)
    o2 = net["cross_stage2"](b, xyz2, a, xyz1)
    out = torch.cat([o1, o2], dim=2)
    pooled = torch.cat((F.adaptive_max_pool1d(out, 1).view(out.size(0), -1), F.adaptive_avg_pool1d(out, 1).view(out.size(0), -1)), 1)
    return net["match_head"](pooled).squeeze(1)


@torch.no_grad()
def ref_match_search(net, h1, h2, xyz1, xyz2, local):
    """ReIDNet.xcorr / xcorr_baseline + get_pooled_feats('both') + match_head (ReIDNet.py:250-264, 444-448)."""
    a = net["cross_stage1"](h1, xyz1, h2, xyz2)
    if local:
        a = net["local_stage1"](a, xyz1)
    a = net["cross_stage2"](a, xyz1, h2, xyz2)
    if local:
        a = net["local_stage2"](a, xyz1)
    pooled = torch.cat((F.adaptive_max_pool1d(a, 1).view(a.size(0), -1), F.adaptive_avg_pool1d(a, 1).view(a.size(0), -1)), 1)
    return net["match_head"](pooled).squeeze(1)


def main_xcorr(R):
    """'xcorr' (local_self_attention stages) and 'xcorr-baseline' match types of the shipped PT configs."""
    for kind, local in (("xcorr", True), ("xcorr-baseline", False)):
        net, sd = build_reference(R, "pt", local=local)
        T, D, N, blist = 3, 4, 128, [128, 64, 32]
        t, d = O.synth_objects(T, N, 0), O.synth_objects(D, N, 1)
        xt, ht = ref_encode(net, "pt", t, blist)
        xd, hd = ref_encode(net, "pt", d, blist)
        pairs = torch.cartesian_prod(torch.arange(T), torch.arange(D))
        logits = ref_match_search(net, ht[pairs[:, 0]], hd[pairs[:, 1]], xt[pairs[:, 0]], xd[pairs[:, 1]], local).reshape(T, D)
        np.savez_compressed(os.path.join(OUT, f"reid_{kind}.npz"), tracks=t.numpy(), dets=d.numpy(), h_t=ht.numpy(),
                            h_d=hd.numpy(), logits=logits.numpy(), weight_checksum=np.float64(checksum(sd)),
                            backbone_list=np.array(blist))
        print(kind, "logits std", float(logits.std()), "checksum", checksum(sd))


def build_image_reference(R, dim=192, dd=64):
    """Reference modules in ImageReIDNet.__init__ construction order (cross_stage1, cross_stage2, cls_head, match_head,
    vis_head, fp_head, downsample; ReIDNet.py:852-859), config reid_image_deit-tiny_point-cat.py."""
    torch.manual_seed(66)
    hp = 2 * dim
    aux = lambda n: torch.nn.Sequential(R.LinearRes(hp, hp, norm='GN', ng=64), torch.nn.Linear(hp, n))
    mods = {}
    mods["cross_stage1"] = R.cross_lin_attn(d_model=dd, nhead=2, attention='linear')
    mods["cross_stage2"] = R.cross_lin_attn(d_model=dd, nhead=2, attention='linear')
    mods["cls_head"] = aux(20)
    mods["match_head"] = torch.nn.Sequential(R.LinearRes(2 * dd, 2 * dd, norm='GN', ng=16), torch.nn.Linear(2 * dd, 1))
    mods["vis_head"] = aux(4)
    mods["fp_head"] = aux(1)
    mods["downsample"] = torch.nn.Sequential(R.LinearRes(dim, 256, norm='GN', ng=32), R.LinearRes(256, 128, norm='GN', ng=16),
                                             torch.nn.Linear(128, dd))
    net = torch.nn.ModuleDict(mods).eval()
    sd = O.perturb_norm_state(net.state_dict())
    net.load_state_dict(sd)
    return net, sd


@torch.no_grad()
def main_image(R):
    """token side of ImageReIDNet: downsample (ReIDNet.py:1276-1277), xcorr_eff with cross_lin_attn (896-912), pooling
    'both' (1147-1155), match head (1057-1066); 198 tokens = DeiT-distilled @224."""
    net, sd = build_image_reference(R)
    dim, dd, S, T, D = 192, 64, 198, 3, 4
    raw = O.synth_tokens(2, dim, S, 0)
    b, c, s = raw.shape
    h_raw = net["downsample"](raw.reshape(-1, c)).reshape(b, dd, s)
    h_t, h_d = O.synth_tokens(T, dd, S, 1), O.synth_tokens(D, dd, S, 2)
    pairs = torch.cartesian_prod(torch.arange(T), torch.arange(D))
    o1, o2 = h_t[pairs[:, 0]], h_d[pairs[:, 1]]
    a, bb = net["cross_stage1"](o1, o2), net["cross_stage1"](o2, o1)
    out = torch.cat([net["cross_stage2"](a, bb), net["cross_stage2"](bb, a)], dim=2)
    pooled = torch.cat((F.adaptive_max_pool1d(out, 1).view(out.size(0), -1), F.adaptive_avg_pool1d(out, 1).view(out.size(0), -1)), 1)
    logits = net["match_head"](pooled).squeeze(1).reshape(T, D)
    np.savez_compressed(os.path.join(OUT, "reid_image_tokens.npz"), raw=raw.numpy(), h_raw=h_raw.numpy(), h_t=h_t.numpy(),
                        h_d=h_d.numpy(), logits=logits.numpy(), weight_checksum=np.float64(checksum(sd)))
    print("image tokens: logits std", float(logits.std()), "checksum", checksum(sd))


def main():
    R = ref_loader.load()
    os.makedirs(OUT, exist_ok=True)
    if "--xcorr-only" in sys.argv:
        return main_xcorr(R)
    if "--image-only" in sys.argv:
        return main_image(R)
    for kind, N, blist, T, D in (("pt", 128, [128, 64, 32], 4, 5), ("pt256", 256, [256, 128, 64], 2, 3),
                                 ("dgcnn", 128, [128, 64, 32], 3, 4), ("pointnet", 128, [128, 64, 32], 4, 4)):
        base = "pt" if kind.startswith("pt") else kind
        net, sd = build_reference(R, base)
        t = O.synth_objects(T, N, 0)
        d = O.synth_objects(D, N, 1)
        xt, ht = ref_encode(net, base, t, blist)
        xd, hd = ref_encode(net, base, d, blist)
        pairs = torch.cartesian_prod(torch.arange(T), torch.arange(D))
        logits = ref_match(net, ht[pairs[:, 0]], hd[pairs[:, 1]], xt[pairs[:, 0]], xd[pairs[:, 1]]).reshape(T, D)
        np.savez_compressed(os.path.join(OUT, f"reid_{kind}.npz"), tracks=t.numpy(), dets=d.numpy(), h_t=ht.numpy(),
                            h_d=hd.numpy(), logits=logits.numpy(), weight_checksum=np.float64(checksum(sd)),
                            backbone_list=np.array(blist))
        print(kind, "h", tuple(ht.shape), "logits std", float(logits.std()), "checksum", checksum(sd))
    # kNN index golden from the reference's own knn_point / dgcnn knn on tie-free input
    p2 = R.pointnet2_utils
    x = O.synth_objects(3, 160, 5)
    idx = p2.knn_point(48, x, x[:, :80])
    xf = torch.randn(2, 64, 96, generator=torch.Generator().manual_seed(3))
    idx_f = R.dgcnn_orig.knn(xf, 20)
    np.savez_compressed(os.path.join(OUT, "knn_torch_path.npz"), xyz=x.numpy(), idx=idx.numpy().astype(np.int32),
                        feat=xf.numpy(), idx_feat=idx_f.numpy().astype(np.int32))
    print("knn golden written")
    main_xcorr(R)
    main_image(R)


if __name__ == "__main__":
    main()
