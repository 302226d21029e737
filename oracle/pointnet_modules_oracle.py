"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the mmdet3d PointNet++ modules
(mmdet3d/ops/pointnet_modules/point_sa_module.py:164-208 BasePointSAModule.forward, point_fp_module.py:39-79
PointFPModule.forward) as plain torch over the op oracle (oracle/ops_oracle.py).

PINNED (tests/test_pointnet_modules_pinned.py, wherever PCREID_REFERENCE_ROOT names the upstream source tree): bit-exact against the reference's own module
files imported unmodified by path (oracle/ref_loader.load_pointnet_modules) -- BasePointSAModule / PointSAModuleMSG /
PointSAModule / build_sa_module, PointFPModule, QueryAndGroup / GroupAll, Points_Sampler / calc_square_dist -- run on CPU with
(a) the compiled CUDA ops replaced by oracle/ops_oracle.py, which is pinned to the reference .cu files on the GPU box, and
(b) mmcv's ConvModule (a third-party dependency that is absent here) replaced by a torch stand-in with mmcv's documented
conv -> norm -> activation order.  The glue restated here: sample -> gather -> for each scale
QueryAndGroup (group_points.py:49-83) -> Conv2d 1x1 / BatchNorm2d (eval) / ReLU -> max (or mean) over the samples -> concat;
samplers D-FPS / F-FPS / FS (furthest_point_sample/points_sampler.py:67-157, utils.py:4-31).
"""
import torch
import torch.nn.functional as F

from . import ops_oracle as OP


def conv_module(sd, p, x):
    """mmcv ConvModule(1x1 Conv2d, BN2d, ReLU) in eval mode; x (B, C, S, k)."""
    x = F.conv2d(x, sd[p + ".conv.weight"], sd.get(p + ".conv.bias"))
    if (p + ".bn.weight") in sd:
        x = F.batch_norm(x, sd[p + ".bn.running_mean"], sd[p + ".bn.running_var"], sd[p + ".bn.weight"], sd[p + ".bn.bias"],
                         False, 0.0, 1e-5)
    return F.relu(x)


def _mlp(sd, p, x):
    i = 0
    while (f"{p}.layer{i}.conv.weight") in sd:
        x = conv_module(sd, f"{p}.layer{i}", x)
        i += 1
    return x


def query_and_group(points_xyz, center_xyz, features, max_radius, sample_num, min_radius=0, use_xyz=True, normalize_xyz=False):
    idx = OP.ball_query(min_radius, max_radius, sample_num, points_xyz, center_xyz)
    xyz_trans = points_xyz.transpose(1, 2).contiguous()
    grouped_xyz = OP.grouping_operation(xyz_trans, idx)
    diff = grouped_xyz - center_xyz.transpose(1, 2).unsqueeze(-1)
    if normalize_xyz:
        diff = diff / max_radius
    if features is not None:
        gf = OP.grouping_operation(features, idx)
        return torch.cat([diff, gf], dim=1) if use_xyz else gf
    return diff


def uniform_resample(idx, sample_num):
    """uniform_sample branch of QueryAndGroup.forward (group_points.py:78-91) restated: per (batch, region) keep the distinct
    indices (torch.unique: ascending) and fill up to sample_num with torch.randint picks among them (host default generator,
    one call per region in (batch, region) order).  -> (idx, unique_cnt (B, S) float32)."""
    idx = idx.clone()
    cnt = torch.zeros((idx.shape[0], idx.shape[1]))
    for b in range(idx.shape[0]):
        for r in range(idx.shape[1]):
            u = torch.unique(idx[b, r, :])
            n = u.shape[0]
            cnt[b, r] = n
            fill = torch.randint(0, n, (sample_num - n,), dtype=torch.long)
            idx[b, r, :] = torch.cat((u, u[fill]))
    return idx, cnt


def query_and_group_full(points_xyz, center_xyz, features, max_radius, sample_num, min_radius=0, use_xyz=True, normalize_xyz=False,
                         uniform_sample=False):
    """QueryAndGroup.forward (group_points.py:49-129) with every return it can be configured to give:
    -> (new_features, grouped_xyz, unique_cnt or None, idx)."""
    if max_radius is None:
        idx = OP.knn(sample_num, points_xyz, center_xyz).transpose(1, 2).contiguous()
    else:
        idx = OP.ball_query(min_radius, max_radius, sample_num, points_xyz, center_xyz)
    cnt = None
    if uniform_sample:
        idx, cnt = uniform_resample(idx, sample_num)
    grouped_xyz = OP.grouping_operation(points_xyz.transpose(1, 2).contiguous(), idx)
    diff = grouped_xyz - center_xyz.transpose(1, 2).unsqueeze(-1)
    if normalize_xyz:
        diff = diff / max_radius
    if features is not None:
        gf = OP.grouping_operation(features, idx)
        nf = torch.cat([diff, gf], dim=1) if use_xyz else gf
    else:
        nf = diff
    return nf, grouped_xyz, cnt, idx


def calc_square_dist_ref(a, b, norm=True):
    """furthest_point_sample/utils.py:4-31 verbatim (torch sum / matmul): what the reference feeds to F-FPS."""
    length_a, length_b, num_channel = a.shape[1], b.shape[1], a.shape[-1]
    a_square = torch.sum(a.unsqueeze(dim=2).pow(2), dim=-1).repeat((1, 1, length_b))
    b_square = torch.sum(b.unsqueeze(dim=1).pow(2), dim=-1).repeat((1, length_a, 1))
    dist = a_square + b_square - 2 * torch.matmul(a, b.transpose(1, 2))
    if norm:
        dist = torch.sqrt(dist) / num_channel
    return dist


def _sample(mod, points, features, npoint, sqdist):
    """DFPS / FFPS / FS samplers (points_sampler.py:107-157)."""
    if mod == "D-FPS":
        return OP.furthest_point_sample(points.contiguous(), npoint)
    f = torch.cat([points, features.transpose(1, 2)], dim=2)
    ffps = OP.furthest_point_sample_with_dist(sqdist(f, f, norm=False).contiguous(), npoint)
    if mod == "F-FPS":
        return ffps
    if mod == "FS":
        return torch.cat([ffps, OP.furthest_point_sample(points.contiguous(), npoint)], dim=1)
    raise ValueError(mod)


def points_sampler(points_xyz, features, num_point, fps_mod_list=("D-FPS",), fps_sample_range_list=(-1,), sqdist=None):
    """Points_Sampler.forward (points_sampler.py:67-104).  sqdist: OP.pairwise_sqdist (the kernel's arithmetic, default) or
    calc_square_dist_ref (the reference's torch ops)."""
    sqdist = sqdist or OP.pairwise_sqdist
    indices, last = [], 0
    for rng, mod, npoint in zip(fps_sample_range_list, fps_mod_list, num_point):
        assert rng < points_xyz.shape[1]
        if rng == -1:
            xyz, feats = points_xyz[:, last:], (features[:, :, last:] if features is not None else None)
        else:
            xyz, feats = points_xyz[:, last:rng], (features[:, :, last:rng] if features is not None else None)
        indices.append(_sample(mod, xyz.contiguous(), feats, npoint, sqdist) + last)
        last += rng
    return torch.cat(indices, dim=1)


def _pool(x, pool_mod):
    """BasePointSAModule._pool_features (point_sa_module.py:144-164)."""
    fn = F.max_pool2d if pool_mod == "max" else F.avg_pool2d
    return fn(x, kernel_size=[1, x.size(3)]).squeeze(-1)


def sa_module_msg(sd, num_point, radii, sample_nums, points_xyz, features=None, indices=None, use_xyz=True, normalize_xyz=False,
                  dilated_group=False, prefix="", pool_mod="max", fps_mod=("D-FPS",), fps_sample_range_list=(-1,), sqdist=None):
    """-> new_xyz, new_features, indices.  sqdist: distance function of the F-FPS / FS samplers (see points_sampler)."""
    xyz_flipped = points_xyz.transpose(1, 2).contiguous()
    if num_point is None:
        g = xyz_flipped.unsqueeze(2)
        if features is not None:
            g = torch.cat([g, features.unsqueeze(2)], dim=1) if use_xyz else features.unsqueeze(2)
        x = _mlp(sd, prefix + "mlps.0", g)
        return None, _pool(x, pool_mod), None
    if indices is None:
        npts = [num_point] if isinstance(num_point, int) else list(num_point)
        indices = points_sampler(points_xyz, features, npts, fps_mod, fps_sample_range_list, sqdist=sqdist)
    new_xyz = OP.gather_points(xyz_flipped, indices).transpose(1, 2).contiguous()
    outs = []
    for i in range(len(radii)):
        mn = radii[i - 1] if (dilated_group and i != 0) else 0
        g = query_and_group(points_xyz, new_xyz, features, radii[i], sample_nums[i], mn, use_xyz, normalize_xyz)
        x = _mlp(sd, f"{prefix}mlps.{i}", g)
        outs.append(_pool(x, pool_mod))
    return new_xyz, torch.cat(outs, dim=1), indices


def fp_module(sd, target, source, target_feats, source_feats, prefix=""):
    if source is not None:
        dist, idx = OP.three_nn(target, source)
        dr = 1.0 / (dist + 1e-8)
        w = dr / torch.sum(dr, dim=2, keepdim=True)
        interp = OP.three_interpolate(source_feats, idx, w)
    else:
        interp = source_feats.expand(*source_feats.size()[0:2], target.size(1))
    x = torch.cat([interp, target_feats], dim=1) if target_feats is not None else interp
    return _mlp(sd, prefix + "mlps", x.unsqueeze(-1)).squeeze(-1)
