"""TEST INFRASTRUCTURE ONLY -- loads the *unmodified* reference leaf modules by path.

Only usable where a checkout of the upstream project (bentherien/point-cloud-reid) is named by the environment variable
``PCREID_REFERENCE_ROOT``; the repository does not contain it.  It is used to
  (1) pin ``oracle/reid_oracle.py`` (our CPU restatement) against the real reference code, and
  (2) generate the committed golden vectors under ``tests/golden/`` (``oracle/make_golden.py``).
Nothing in the product package, ``bench.py`` or the ``-m gpu`` tests may import this file.

``load()`` imports every leaf file holding the arithmetic of the path; ``load_reidnet()`` adds
``mmdet3d/models/ReIDNet.py`` itself (the real ReIDNet / ImageReIDNet classes; mmcv / mmdet / pytorch3d are
absent, so their registry / base class / chamfer loss are stand-ins -- see its docstring).  The leaf files
need three non-invasive shims, none of which touches the reference tree:
  * ``fractions.gcd`` (removed in py3.9) is aliased to ``math.gcd`` before ``lanegcn_nets.py`` loads
    (``lanegcn_nets.py:6``);
  * the module-global ``torch`` of ``dgcnn_orig`` / ``attention`` is replaced by a proxy whose
    ``.device('cuda')`` returns the CPU device (``dgcnn_orig.py:37``, ``attention.py:115,139``);
  * a fake parent package so the relative imports of ``backbone_net.py`` resolve.
"""
import importlib.util
import math
import os
import sys
import types

REF_ROOT = os.environ.get("PCREID_REFERENCE_ROOT", "")
MISSING = "needs the upstream point-cloud-reid source tree, named by PCREID_REFERENCE_ROOT (not part of this repository)"
_MODELS = os.path.join(REF_ROOT, "mmdet3d", "models")
_PKG = "_pcreid_ref_models"


def available():
    return bool(REF_ROOT) and os.path.isdir(_MODELS)


class _TorchProxy(types.ModuleType):
    """Forwards everything to torch but maps device('cuda') to CPU."""

    def __init__(self, real):
        super().__init__("torch")
        object.__setattr__(self, "_real", real)

    def __getattr__(self, name):
        return getattr(object.__getattribute__(self, "_real"), name)

    def device(self, *a, **k):
        real = object.__getattribute__(self, "_real")
        if a and isinstance(a[0], str) and a[0].startswith("cuda"):
            return real.device("cpu")
        return real.device(*a, **k)


def _load(name):
    full = f"{_PKG}.{name}"
    if full in sys.modules:
        return sys.modules[full]
    spec = importlib.util.spec_from_file_location(full, os.path.join(_MODELS, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[full] = mod
    spec.loader.exec_module(mod)
    return mod


def load():
    """Returns a namespace with the reference classes used on the hot path."""
    if not available():
        raise RuntimeError(f"reference tree not found: PCREID_REFERENCE_ROOT={REF_ROOT!r}")
    import fractions
    if not hasattr(fractions, "gcd"):
        fractions.gcd = math.gcd
    import torch
    if _PKG not in sys.modules:
        pkg = types.ModuleType(_PKG)
        pkg.__path__ = [_MODELS]
        sys.modules[_PKG] = pkg
    p2 = _load("pointnet2_utils")
    bb = _load("backbone_net")
    dg = _load("dgcnn_orig")
    pn = _load("pointnet")
    at = _load("attention")
    lg = _load("lanegcn_nets")
    proxy = _TorchProxy(torch)
    dg.torch = proxy
    at.torch = proxy
    ns = types.SimpleNamespace(
        pointnet2_utils=p2, backbone_net=bb, dgcnn_orig=dg, pointnet=pn, attention=at, lanegcn_nets=lg,
        Pointnet_Backbone=bb.Pointnet_Backbone, DGCNN=dg.DGCNN, PointNet=pn.PointNet,
        corss_attention=at.corss_attention, LinearRes=lg.LinearRes, local_self_attention=at.local_self_attention,
        cross_lin_attn=at.cross_lin_attn,
    )
    return ns


# ------------------------------------------------------------------------------------------------------------------
# mmdet3d PointNet++ module family (SURVEY 8f row 3): the reference's own module glue on CPU
# ------------------------------------------------------------------------------------------------------------------
_OPS = os.path.join(REF_ROOT, "mmdet3d", "ops")
_OPS_PKG = "_pcreid_ref_ops"


def pointnet_modules_available():
    return bool(REF_ROOT) and os.path.isdir(os.path.join(_OPS, "pointnet_modules"))


def load_pointnet_modules():
    """Loads the *unmodified* reference files ops/pointnet_modules/{builder,point_sa_module,point_fp_module}.py,
    ops/group_points/group_points.py (QueryAndGroup, GroupAll) and ops/furthest_point_sample/{points_sampler,utils}.py by path
    and runs their Python glue on CPU.  What is NOT the reference's code underneath, and why:
      * the compiled CUDA ops (`*_ext` pybind modules: FPS, ball query, grouping, gather, three_nn, three_interpolate) are
        replaced by the CPU restatements of oracle/ops_oracle.py, themselves pinned bit-exact against the reference .cu
        files on the GPU box (tests/test_gpu_ops.py);
      * mmcv is absent: `mmcv.cnn.ConvModule` is a torch stand-in with mmcv's documented order conv -> norm -> activation and
        its `conv` / `bn` attribute names, `mmcv.runner.BaseModule` is `nn.Module` + a stored `init_cfg`, `force_fp32` an identity decorator,
        `mmcv.utils.Registry` a dict-backed registry; PAConv is a placeholder class (never instantiated).
    Nothing is written into the reference tree; the temporary `mmcv` / `mmdet3d` entries in sys.modules are removed again."""
    import torch
    from torch import nn
    from . import ops_oracle as OP

    class ConvModule(nn.Module):
        def __init__(self, in_channels, out_channels, kernel_size=1, stride=1, conv_cfg=None, norm_cfg=None,
                     act_cfg=dict(type="ReLU"), bias="auto", **kw):
            super().__init__()
            conv = {"Conv2d": nn.Conv2d, "Conv1d": nn.Conv1d}[(conv_cfg or dict(type="Conv2d"))["type"]]
            self.with_norm, self.with_activation = norm_cfg is not None, act_cfg is not None
            if bias == "auto":
                bias = not self.with_norm
            self.conv = conv(in_channels, out_channels, kernel_size, stride=stride, bias=bias)
            if self.with_norm:
                self.bn = {"BN2d": nn.BatchNorm2d, "BN1d": nn.BatchNorm1d, "BN": nn.BatchNorm2d}[norm_cfg["type"]](out_channels)
            if self.with_activation:
                self.activate = nn.ReLU(inplace=True)

        def forward(self, x):
            x = self.conv(x)
            if self.with_norm:
                x = self.bn(x)
            return self.activate(x) if self.with_activation else x

    class Registry:
        def __init__(self, name):
            self.name, self.module_dict = name, {}

        def register_module(self, name=None, **kw):
            def deco(cls):
                self.module_dict[name or cls.__name__] = cls
                return cls
            return deco

        def get(self, key):
            return self.module_dict.get(key)

        def __contains__(self, key):
            return key in self.module_dict

    class BaseModule(nn.Module):          # mmcv.runner.BaseModule: nn.Module + an init_cfg it only stores
        def __init__(self, init_cfg=None):
            super().__init__()
            self.init_cfg = init_cfg

    def force_fp32(*a, **k):
        return lambda fn: fn

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    def load(full, path, package=None):
        spec = importlib.util.spec_from_file_location(full, path)
        m = importlib.util.module_from_spec(spec)
        if package:
            m.__package__ = package
        sys.modules[full] = m
        spec.loader.exec_module(m)
        return m

    saved = {k: sys.modules.get(k) for k in ("mmcv", "mmcv.cnn", "mmcv.runner", "mmcv.utils", "mmdet3d", "mmdet3d.ops")}
    created = []
    try:
        sys.modules["mmcv"] = mod("mmcv")
        sys.modules["mmcv.cnn"] = mod("mmcv.cnn", ConvModule=ConvModule)
        sys.modules["mmcv.runner"] = mod("mmcv.runner", BaseModule=BaseModule, force_fp32=force_fp32)
        sys.modules["mmcv.utils"] = mod("mmcv.utils", Registry=Registry)

        def pkg(name, path):
            p = types.ModuleType(name)
            p.__path__ = [path]
            sys.modules[name] = p
            created.append(name)
            return p

        pkg(_OPS_PKG, _OPS)
        i32 = lambda t: t.to(torch.int32)
        # the compiled ops -> CPU restatements with the reference wrappers' signatures
        bq = pkg(f"{_OPS_PKG}.ball_query", os.path.join(_OPS, "ball_query"))
        bq.ball_query = lambda mn, mx, ns, xyz, cen: i32(OP.ball_query(mn, mx, ns, xyz, cen))
        kn = pkg(f"{_OPS_PKG}.knn", os.path.join(_OPS, "knn"))
        kn.knn = lambda k, xyz, cen=None, transposed=False: i32(OP.knn(k, xyz, cen, transposed))
        gp = pkg(f"{_OPS_PKG}.group_points", os.path.join(_OPS, "group_points"))
        sys.modules[f"{_OPS_PKG}.group_points.group_points_ext"] = mod("group_points_ext")
        created.append(f"{_OPS_PKG}.group_points.group_points_ext")
        gpm = load(f"{_OPS_PKG}.group_points.group_points", os.path.join(_OPS, "group_points", "group_points.py"),
                   f"{_OPS_PKG}.group_points")
        created.append(f"{_OPS_PKG}.group_points.group_points")
        gpm.grouping_operation = lambda feats, idx: OP.grouping_operation(feats, idx)     # module global used by QueryAndGroup
        fps = pkg(f"{_OPS_PKG}.furthest_point_sample", os.path.join(_OPS, "furthest_point_sample"))
        sys.modules[f"{_OPS_PKG}.furthest_point_sample.furthest_point_sample"] = mod(
            "furthest_point_sample", furthest_point_sample=lambda p, n: i32(OP.furthest_point_sample(p, n)),
            furthest_point_sample_with_dist=lambda d, n: i32(OP.furthest_point_sample_with_dist(d, n)))
        created.append(f"{_OPS_PKG}.furthest_point_sample.furthest_point_sample")
        utils = load(f"{_OPS_PKG}.furthest_point_sample.utils", os.path.join(_OPS, "furthest_point_sample", "utils.py"),
                     f"{_OPS_PKG}.furthest_point_sample")
        created.append(f"{_OPS_PKG}.furthest_point_sample.utils")
        ps = load(f"{_OPS_PKG}.furthest_point_sample.points_sampler", os.path.join(_OPS, "furthest_point_sample", "points_sampler.py"),
                  f"{_OPS_PKG}.furthest_point_sample")
        created.append(f"{_OPS_PKG}.furthest_point_sample.points_sampler")

        class PAConv(nn.Module):          # placeholder: only isinstance-checked by the SA module
            pass

        gather = lambda feats, idx: OP.gather_points(feats, idx)
        sys.modules["mmdet3d"] = mod("mmdet3d")
        sys.modules["mmdet3d.ops"] = mod(
            "mmdet3d.ops", GroupAll=gpm.GroupAll, QueryAndGroup=gpm.QueryAndGroup, PAConv=PAConv, Points_Sampler=ps.Points_Sampler,
            gather_points=gather, three_nn=lambda t, s: OP.three_nn(t, s),
            three_interpolate=lambda f, i, w: OP.three_interpolate(f, i, w))
        pm = pkg(f"{_OPS_PKG}.pointnet_modules", os.path.join(_OPS, "pointnet_modules"))
        builder = load(f"{_OPS_PKG}.pointnet_modules.builder", os.path.join(_OPS, "pointnet_modules", "builder.py"),
                       f"{_OPS_PKG}.pointnet_modules")
        sa = load(f"{_OPS_PKG}.pointnet_modules.point_sa_module", os.path.join(_OPS, "pointnet_modules", "point_sa_module.py"),
                  f"{_OPS_PKG}.pointnet_modules")
        fp = load(f"{_OPS_PKG}.pointnet_modules.point_fp_module", os.path.join(_OPS, "pointnet_modules", "point_fp_module.py"),
                  f"{_OPS_PKG}.pointnet_modules")
        created += [f"{_OPS_PKG}.pointnet_modules.builder", f"{_OPS_PKG}.pointnet_modules.point_sa_module",
                    f"{_OPS_PKG}.pointnet_modules.point_fp_module"]
        return types.SimpleNamespace(PointSAModuleMSG=sa.PointSAModuleMSG, PointSAModule=sa.PointSAModule,
                                     PointFPModule=fp.PointFPModule, build_sa_module=builder.build_sa_module,
                                     Points_Sampler=ps.Points_Sampler, calc_square_dist=utils.calc_square_dist,
                                     QueryAndGroup=gpm.QueryAndGroup, GroupAll=gpm.GroupAll)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# ------------------------------------------------------------------------------------------------------------------
# crop -> centre -> resample front-end (SURVEY 8f row 2): the reference's own pc_utils.py + box structures on CPU
# ------------------------------------------------------------------------------------------------------------------
_STRUCTS = os.path.join(REF_ROOT, "mmdet3d", "core", "bbox", "structures")
_PC_UTILS = os.path.join(_MODELS, "trackers", "deprecated", "pc_utils.py")


def frontend_available():
    return bool(REF_ROOT) and os.path.isdir(_STRUCTS) and os.path.exists(_PC_UTILS)


def load_frontend():
    """Loads the *unmodified* reference files models/trackers/deprecated/pc_utils.py (interpolate_per_frame,
    get_input_batch, get_affine_torch) and core/bbox/structures/{base_box3d,utils,depth_box3d,lidar_box3d,cam_box3d,
    box_3d_mode}.py (DepthInstance3DBoxes, Box3DMode.convert) by path and runs them on CPU.  Stand-ins, none of which touches
    the reference tree:
      * pytorch3d (absent; the reference pins no version): `Pointclouds(list).points_padded()` = zero padding to the longest
        cloud, `transforms.axis_angle_to_matrix` = quaternion_to_matrix(axis_angle_to_quaternion(.)) as published in
        pytorch3d 0.7 (rotation_conversions.py);
      * the compiled ops: `mmdet3d.ops.points_in_boxes_batch` -> oracle.frontend_oracle.pib_kernel_lidar (restatement of
        points_in_boxes_cuda.cu, pinned against that .cu on the GPU box); iou3d / roiaware extensions and BasePoints are
        placeholders (never called on this path)."""
    import importlib
    import torch
    from . import frontend_oracle as FO

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    class Pointclouds:
        def __init__(self, points):
            self._p = list(points)

        def points_padded(self):
            n = max([x.shape[0] for x in self._p] + [0])
            out = torch.zeros((len(self._p), n, 3), dtype=torch.float32)
            for i, x in enumerate(self._p):
                out[i, :x.shape[0]] = x
            return out

    def quaternion_to_matrix(quaternions):
        r, i, j, k = torch.unbind(quaternions, -1)
        two_s = 2.0 / (quaternions * quaternions).sum(-1)
        o = torch.stack((1 - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r),
                         two_s * (i * j + k * r), 1 - two_s * (i * i + k * k), two_s * (j * k - i * r),
                         two_s * (i * k - j * r), two_s * (j * k + i * r), 1 - two_s * (i * i + j * j)), -1)
        return o.reshape(quaternions.shape[:-1] + (3, 3))

    def axis_angle_to_quaternion(axis_angle):
        angles = torch.norm(axis_angle, p=2, dim=-1, keepdim=True)
        half_angles = angles * 0.5
        small = angles.abs() < 1e-6
        k = torch.empty_like(angles)
        k[~small] = torch.sin(half_angles[~small]) / angles[~small]
        k[small] = 0.5 - (angles[small] * angles[small]) / 48
        return torch.cat([torch.cos(half_angles), axis_angle * k], dim=-1)

    def points_in_boxes_batch(points, boxes):
        assert points.shape[0] == boxes.shape[0] == 1
        inside, _ = FO.pib_kernel_lidar(boxes[0].numpy(), points[0].numpy())
        return torch.from_numpy(inside.T.astype("int32")).unsqueeze(0)             # (B, M, T)

    names = ("pytorch3d", "pytorch3d.transforms", "pytorch3d.structures", "pytorch3d.structures.pointclouds", "mmdet3d",
             "mmdet3d.core", "mmdet3d.core.points", "mmdet3d.ops", "mmdet3d.ops.iou3d", "mmdet3d.ops.roiaware_pool3d",
             "nuscenes", "nuscenes.utils", "nuscenes.utils.geometry_utils", "torchvision", "torchvision.transforms")
    saved = {k: sys.modules.get(k) for k in names}
    try:
        sys.modules["pytorch3d"] = mod("pytorch3d")
        sys.modules["pytorch3d.transforms"] = mod("pytorch3d.transforms", quaternion_to_matrix=quaternion_to_matrix,
                                                  axis_angle_to_matrix=lambda aa: quaternion_to_matrix(axis_angle_to_quaternion(aa)))
        sys.modules["pytorch3d"].transforms = sys.modules["pytorch3d.transforms"]
        sys.modules["pytorch3d.structures"] = mod("pytorch3d.structures")
        sys.modules["pytorch3d.structures.pointclouds"] = mod("pytorch3d.structures.pointclouds", Pointclouds=Pointclouds)
        # module-level imports of the image-crop half of pc_utils.py (lines 112-122), unused on this path
        for n, attrs in (("nuscenes", {}), ("nuscenes.utils", {}), ("nuscenes.utils.geometry_utils", dict(BoxVisibility=type("BoxVisibility", (), dict(ANY=1, ALL=0, NONE=2))))):
            sys.modules[n] = mod(n, **attrs)
        try:
            import torchvision.transforms  # noqa: F401
        except Exception:
            sys.modules["torchvision"] = mod("torchvision")
            sys.modules["torchvision.transforms"] = mod("torchvision.transforms", ToTensor=None)
        sys.modules["mmdet3d"] = mod("mmdet3d")
        sys.modules["mmdet3d.core.points"] = mod("mmdet3d.core.points", BasePoints=type("BasePoints", (), {}))
        sys.modules["mmdet3d.ops"] = mod("mmdet3d.ops", points_in_boxes_batch=points_in_boxes_batch)
        sys.modules["mmdet3d.ops.iou3d"] = mod("mmdet3d.ops.iou3d", iou3d_cuda=None)
        sys.modules["mmdet3d.ops.roiaware_pool3d"] = mod("mmdet3d.ops.roiaware_pool3d", points_in_boxes_gpu=None)
        pkg = "_pcreid_ref_structs"
        if pkg not in sys.modules:
            p = types.ModuleType(pkg)
            p.__path__ = [_STRUCTS]                 # a bare package: the reference __init__.py (which pulls in mmcv) is not run
            sys.modules[pkg] = p
        depth = importlib.import_module(f"{pkg}.depth_box3d")
        b3d = importlib.import_module(f"{pkg}.box_3d_mode")
        sys.modules["mmdet3d.core"] = mod("mmdet3d.core", DepthInstance3DBoxes=depth.DepthInstance3DBoxes)
        spec = importlib.util.spec_from_file_location("_pcreid_ref_pc_utils", _PC_UTILS)
        pcu = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(pcu)
        return types.SimpleNamespace(pc_utils=pcu, DepthInstance3DBoxes=depth.DepthInstance3DBoxes, Box3DMode=b3d.Box3DMode,
                                     interpolate_per_frame=pcu.interpolate_per_frame, get_input_batch=pcu.get_input_batch)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# ------------------------------------------------------------------------------------------------------------------
# all-pairs driver + feature bank (SURVEY 8f row 1): the reference's own deprecated tracker files on CPU
# ------------------------------------------------------------------------------------------------------------------
_TRK = os.path.join(_MODELS, "trackers", "deprecated")


def tracker_available():
    return bool(REF_ROOT) and os.path.exists(os.path.join(_TRK, "tracking_point_reid.py")) and os.path.exists(os.path.join(_TRK, "tracking_feature_set.py"))


def load_tracker():
    """Loads the *unmodified* reference files trackers/deprecated/tracking_point_reid.py (get_labels_to_compare,
    PointReidentifier) and tracking_feature_set.py (PointFeatureSet) by path.  Stand-ins: the mmcv-backed `TRACKERS` registry and
    `builder.build_tracker` of mmdet3d.models (a dict-backed registry), `mmdet3d.models.trackers.pc_utils` (placeholders: the
    crop helpers are pinned separately by load_frontend) and `mmdet3d.datasets.utils.MatchingEval` (a placeholder, unused)."""
    reg = {}

    class _Registry:
        def register_module(self, name=None, **kw):
            def deco(cls):
                reg[name or cls.__name__] = cls
                return cls
            return deco

    def build_tracker(cfg):
        cfg = dict(cfg)
        return reg[cfg.pop("type")](**cfg)

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    names = ("mmdet3d", "mmdet3d.models", "mmdet3d.models.trackers", "mmdet3d.models.trackers.pc_utils", "mmdet3d.datasets",
             "mmdet3d.datasets.utils")
    saved = {k: sys.modules.get(k) for k in names}
    try:
        builder = mod("mmdet3d.models.builder", build_tracker=build_tracker)
        sys.modules["mmdet3d"] = mod("mmdet3d")
        sys.modules["mmdet3d.models"] = mod("mmdet3d.models", TRACKERS=_Registry(), builder=builder)
        sys.modules["mmdet3d.models.trackers"] = mod("mmdet3d.models.trackers")
        sys.modules["mmdet3d.models.trackers.pc_utils"] = mod("mmdet3d.models.trackers.pc_utils", get_crops_per_image=None,
                                                              interpolate_per_frame=None, get_input_batch=None)
        sys.modules["mmdet3d.datasets"] = mod("mmdet3d.datasets")
        sys.modules["mmdet3d.datasets.utils"] = mod("mmdet3d.datasets.utils", MatchingEval=None)
        out = {}
        for name in ("tracking_feature_set", "tracking_point_reid"):
            spec = importlib.util.spec_from_file_location(f"_pcreid_ref_{name}", os.path.join(_TRK, name + ".py"))
            m = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(m)
            out[name] = m
        return types.SimpleNamespace(get_labels_to_compare=out["tracking_point_reid"].get_labels_to_compare,
                                     PointReidentifier=out["tracking_point_reid"].PointReidentifier,
                                     PointFeatureSet=out["tracking_feature_set"].PointFeatureSet)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


# ------------------------------------------------------------------------------------------------------------------
# the reference's ReIDNet / ImageReIDNet classes themselves (mmdet3d/models/ReIDNet.py), on CPU
# ------------------------------------------------------------------------------------------------------------------
def load_reidnet():
    """Loads the *unmodified* reference file mmdet3d/models/ReIDNet.py by path (after load(), which provides the leaf modules of
    its relative imports under the fake parent package) and returns its classes: ReIDNet, ReIDNetCosine, ImageReIDNet and the
    module factory (module_obj, build_module, build_sequential).  Stand-ins for what is absent here, none of which carries
    arithmetic of the path:
      * `mmdet3d.models.FUSIONMODELS` (an mmcv Registry)  -> a dict-backed registry with `register_module()`;
      * `mmdet.models.BaseDetector`                      -> `nn.Module` (the reference only inherits forward dispatch from it);
      * `pytorch3d.loss.chamfer_distance`                -> a placeholder (training-only shape loss);
      * `transformers` is installed and imported for real (HuggingFace checkpoints are NOT downloaded: ImageReIDNet's
        `get_image_model` must be monkey-patched by the caller)."""
    import torch
    from torch import nn
    ns = load()

    class _Registry:
        def __init__(self):
            self.module_dict = {}

        def register_module(self, name=None, **kw):
            def deco(cls):
                self.module_dict[name or cls.__name__] = cls
                return cls
            return deco

    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        return m

    names = ("mmdet3d", "mmdet3d.models", "mmdet", "mmdet.models", "pytorch3d", "pytorch3d.loss")
    saved = {k: sys.modules.get(k) for k in names}
    try:
        reg = _Registry()
        sys.modules["mmdet3d"] = mod("mmdet3d")
        sys.modules["mmdet3d.models"] = mod("mmdet3d.models", FUSIONMODELS=reg)
        sys.modules["mmdet"] = mod("mmdet")
        sys.modules["mmdet.models"] = mod("mmdet.models", BaseDetector=nn.Module)
        sys.modules["pytorch3d"] = mod("pytorch3d")
        sys.modules["pytorch3d.loss"] = mod("pytorch3d.loss", chamfer_distance=None)
        m = _load("ReIDNet")
        proxy = _TorchProxy(torch)
        m.torch = proxy                   # torch.device('cuda') literals -> CPU, as for dgcnn_orig / attention
        ns.ReIDNet_module = m
        ns.ReIDNet, ns.ReIDNetCosine, ns.ImageReIDNet = m.ReIDNet, m.ReIDNetCosine, m.ImageReIDNet
        ns.module_obj, ns.build_module, ns.build_sequential = m.module_obj, m.build_module, m.build_sequential
        ns.FUSIONMODELS = reg
        return ns
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
