"""ReIDNet -- siamese point-set encoder + match head (mmdet3d/models/ReIDNet.py:111-167 ctor, 189-212
forward / forward_inference, 231-247 xcorr_eff, 311-332 siamese_forward, 444-462 match_forward_inference,
526-534 get_pooled_feats, 637-689 forward_test), inference path only, on the pcreid CUDA kernels.

New relative to the reference: ``match_all_pairs`` scores the whole track x detection matrix the way the
deprecated tracker did (trackers/deprecated/tracking_point_reid.py:95-116) but without materialising
``feat[pairs[:, 0]]`` / ``feat[pairs[:, 1]]``: everything that depends on one object only (stage-1 queries,
key/value summaries, position codes) is computed once per object and gathered through index maps.
"""
import copy

import os

import torch
from torch import nn

from .. import kernels as K
from .attention import corss_attention, cross_lin_attn, local_self_attention
from .backbone_net import Pointnet_Backbone
from .builder import FUSIONMODELS
from .dgcnn_orig import DGCNN
from .lanegcn_nets import LinearRes
from .pointnet import PointNet

module_obj = {
    'Linear': nn.Linear, 'ReLU': nn.ReLU, 'LSTM': nn.LSTM, 'GroupNorm': nn.GroupNorm, 'Embedding': nn.Embedding,
    'LayerNorm': nn.LayerNorm, 'LinearRes': LinearRes, 'Pointnet_Backbone': Pointnet_Backbone,
    'corss_attention': corss_attention, 'Conv1d': nn.Conv1d, 'Conv2d': nn.Conv2d, 'BatchNorm1d': nn.BatchNorm1d,
    'Sigmoid': nn.Sigmoid, 'dgcnn': DGCNN, 'PointNet': PointNet, 'local_self_attention': local_self_attention,
    'cross_lin_attn': cross_lin_attn,
}
_OUT_OF_SCOPE = ('PostRes',)   # lanegcn residual block no shipped ReID config instantiates


def build_module(cfg):
    """ReIDNet.py:78-87 (without mutating the caller's cfg)."""
    if cfg is None or cfg == {}:
        return None
    if isinstance(cfg, list):
        return build_sequential(cfg)
    cfg = dict(cfg)
    typ = cfg.pop('type')
    if typ in _OUT_OF_SCOPE:
        raise NotImplementedError(f"module type '{typ}' is outside the accelerated hot path")
    return module_obj[typ](**cfg)


def build_sequential(module_list):
    if module_list is None or module_list == {}:
        return None
    return nn.Sequential(*[build_module(c) for c in module_list])


def _i32(t):
    return t.to(torch.int32).contiguous()


@FUSIONMODELS.register_module()
class ReIDNet(nn.Module):
    def __init__(self, hidden_size, backbone, cls_head, match_head, shape_head, fp_head, downsample,
                 cross_stage1, local_stage1, cross_stage2, local_stage2, match_type='xcorr', pool_type='max', combine='cat',
                 compute_summary=True, train_cfg=None, test_cfg=None, backbone_list=[512, 256, 128], use_dgcnn=False,
                 losses_to_use=dict(kl=True, match=True, cls=True, shape=True, fp=True, dense=False), output_sequence_size=32,
                 alpha=dict(kl=1, match=1, cls=1, shape=1, fp=1, triplet=1, dense=1), triplet_sample_num=5,
                 triplet_loss=dict(margin=0.2, p=2), eval_only=False, use_o=False, eval_flip=False):
        super().__init__()
        self.eval_only = eval_only
        self.hidden_size = hidden_size
        self.match_type = match_type
        self.backbone = build_module(backbone)
        self.cls_head = build_module(cls_head)
        self.match_head = build_module(match_head)
        self.shape_head = build_module(shape_head)
        self.fp_head = build_module(fp_head)
        self.downsample = build_module(downsample)
        self.cross_stage1 = build_module(cross_stage1)
        self.local_stage1 = build_module(local_stage1)
        self.cross_stage2 = build_module(cross_stage2)
        self.local_stage2 = build_module(local_stage2)
        self.losses_to_use = dict(kl=False, match=True, cls=False, shape=False, fp=False, dense=False)
        self.losses_to_use.update(losses_to_use)
        self.backbone_list = backbone_list
        self.output_sequence_size = output_sequence_size
        self.pool_type = pool_type
        self.maxpool = nn.MaxPool1d(self.output_sequence_size)
        self.bce = nn.BCEWithLogitsLoss()
        self.alpha = alpha
        self.use_o = use_o
        self.eval_flip = eval_flip
        self.verbose = False
        self.sampling = None
        self.compute_summary = compute_summary
        self.use_dgcnn = use_dgcnn
        self.combine = combine
        # 'parity': fp32 kernels (logits within 1e-4 of the reference); 'parity_tc' / 'fast': fused tcgen05 matcher with
        # fp16 / bf16 operands where the configuration allows it (d_model 64, 2 heads, point-cat + both pooling)
        self.match_mode = 'parity'
        self.parity_tc_fp_blocks = False   # True: FP_SA blocks also run as tf32 tcgen05 kernels in 'parity_tc' mode (see set_mode)
        self.parity_tc_x3 = False   # 'parity_tc': K < 256 contractions on the 3 x tf32 kernel instead of the FFMA kernel (see _tc_linear)
        self.tc_encoder = True      # in the tensor-core modes the encoder's 1x1 convs / Linears run as tf32 tcgen05 GEMMs
        self.head_x3 = os.environ.get("PCREID_HEAD_X3", "1") != "0"   # tensor-core modes: match head on the 3 x tf32 GEMM (see _head_cn)
        self._fused = {}
        # encode() replays a captured CUDA graph per (shape, mode, weights version): the ~90 launches of one encoder pass
        # are issued by the GPU front-end instead of by ~90 Python -> ctypes -> cudaLaunchKernel round trips
        self.cuda_graphs = False
        self._graphs = {}
        if self.match_type not in ('xcorr_eff', 'concat', 'xcorr', 'xcorr-baseline'):
            raise NotImplementedError(f"match_type '{match_type}' is outside the accelerated hot path "
                                      "(shipped point configs use 'xcorr_eff'; the baseline uses 'concat')")

    TC_MODES = ('parity_tc', 'fast')

    def set_mode(self, mode):
        """'parity': fp32 FFMA kernels everywhere (|dlogit| <= 1e-4).
        'parity_x3': the parity path with every Linear / 1x1 conv the TMA-staged GEMM can serve on the tensor cores at fp32-grade
        accuracy (pcreid_cn_linear_tma_x3: operands split hi + lo, three kind::tf32 MMAs per K step; ~1e-6 relative to the FFMA
        kernel, same 1e-4 gate) -- the strict-parity mode on tcgen05.
        'parity_tc': the contractions on the tensor cores at an 11-bit significand -- tcgen05 kind::tf32 SA shared MLPs and
        Self_Attention blocks in the encoder (operands pre-rounded to tf32), fused tcgen05 matcher with fp16 operands -- fp32
        accumulation and norms (|dlogit| <= 5e-3, the tf32 gate of SURVEY.md 8d).  The three feature-propagation blocks
        (FP_SA), whose output IS the embedding, stay on the fp32 kernels in this mode unless `parity_tc_fp_blocks` is set:
        measured (scripts/encoder_error_probe.py, profiles/r02_parity_error_budget.md) they alone cost ~1 % of raw top-1
        agreement on the random-init logits (top-2 gap median 5e-3) for 3 % of the step time.
        'fast': every block on the tensor cores, bf16 matcher operands (|dlogit| <= 3e-2)."""
        assert mode in ('parity', 'parity_x3') + self.TC_MODES
        from .pointnet2_utils import FP_SA
        self.match_mode = mode
        for m in self.modules():
            if hasattr(m, 'tc_mode'):
                m.tc_mode = mode in self.TC_MODES and not (mode == 'parity_tc' and isinstance(m, FP_SA) and not self.parity_tc_fp_blocks)
        return self

    def _tc_linear(self):
        """tcgen05 GEMMs for the 1x1 convs / Linears outside the fused kernels: 'fast': every contraction single-pass tf32;
        'parity_tc': K >= 256 single-pass tf32 (the set its error budget was measured with), the rest on the FFMA kernel -- or, with
        `parity_tc_x3`, fp32-grade 3 x tf32 (encode 12.2 -> 10.6 ms per 2048 objects; measured raw top-1 0.982 instead of 0.990 on the
        bench's 384 x 256 block: the near-tied rows follow whichever rounding is closest to the oracle's sequential fp32 sums);
        'parity_x3': everything fp32-grade 3 x tf32; 'parity': none (FFMA kernels)."""
        mode = self.match_mode
        if mode == 'parity_x3':
            # 'xcorr': the matcher's local stages run a feature-space kNN on (functions of) the embeddings; a 1e-6 difference flips
            # near-tied neighbours, which the 1e-4 gate does not absorb -> that configuration stays on the FFMA kernels end to end
            return K.tensor_core_linear(self.tc_encoder and self.match_type != 'xcorr', min_k=1 << 30, x3=True)
        return K.tensor_core_linear(mode in self.TC_MODES and self.tc_encoder, min_k=32 if mode == 'fast' else 256,
                                    x3=self.parity_tc_x3 and mode == 'parity_tc')

    def _tc_match(self, fused):
        """the matcher's Linears outside the fused kernels (per-object preparation; the whole cross-attention chain for shapes
        the fused matcher does not cover: d_model = 128, 'xcorr'): single-pass tf32 in 'fast' mode and, when the fused matcher is
        not in use, in 'parity_tc' mode; around the fused matcher 'parity_tc' keeps the FFMA kernels (fp32-grade 3 x tf32 with
        `parity_tc_x3`); fp32-grade 3 x tf32 everywhere in 'parity_x3'.  The match head always runs on the fp32 kernels."""
        mode = self.match_mode
        if mode == 'parity_x3' and self.match_type == 'xcorr':
            # the local stages run a feature-space kNN on the cross-attended features: a 1e-6 difference flips near-tied neighbours
            return K.tensor_core_linear(False)
        if mode == 'fast' or (mode == 'parity_tc' and not fused):
            return K.tensor_core_linear(True, min_k=32)
        return K.tensor_core_linear(mode == 'parity_x3' or (mode == 'parity_tc' and self.parity_tc_x3), min_k=1 << 30, x3=True)

    def invalidate_packed(self):
        """forget every packed / BN-folded / operand-image weight copy and captured CUDA graph (see _packing.invalidate_packed:
        needed only after parameters were written through `.data`, which no version counter records)."""
        from ._packing import invalidate_packed
        invalidate_packed(self)
        self._fused.clear()
        self._graphs.clear()
        K._W_IMAGES.clear()
        return self

    def fused_matcher(self):
        """the fused tcgen05 matcher of the current tensor-core mode (one per operand format)"""
        from . import fused_pairs
        fmt = fused_pairs.FMT_F16 if self.match_mode == 'parity_tc' else fused_pairs.FMT_BF16
        if fmt not in self._fused:
            self._fused[fmt] = fused_pairs.FusedXcorr(self, fmt)
        return self._fused[fmt]

    # ------------------------------------------------------------------ encoders
    def _encode(self, pts):
        """pts (B, N, 3) -> (xyz (B, N, 3), h (B, C, N)); applies the per-point `downsample` when use_dgcnn is set
        (DGCNN and the shipped PointNet config), exactly as siamese_forward does (ReIDNet.py:316-328)."""
        pts = pts.float().contiguous()
        if self.use_dgcnn or isinstance(self.backbone, (DGCNN, PointNet)):
            _, h = self.backbone(pts.permute(0, 2, 1).contiguous(), self.backbone_list)
            # the reference applies `downsample` in its use_dgcnn branch only (ReIDNet.py:316-324); its
            # `type(self.backbone) == PointNet` branch (:325-328) returns the backbone's raw channel map
            if self.use_dgcnn and self.downsample is not None:
                for m in self.downsample:
                    if isinstance(m, LinearRes):
                        h = m.forward_cn(h)
                    elif isinstance(m, nn.Linear):
                        h = K.cn_linear(h, _kmajor_cached(m), bias=_bias_cached(m))
                    else:
                        raise NotImplementedError(type(m))
            return pts, h
        return self.backbone(pts, self.backbone_list)

    def encode(self, pts):
        """public inference entry: pts (B, N, 3) -> (xyz (B, N, 3), per-point embedding (B, C, N))."""
        with torch.no_grad(), self._tc_linear():
            if self.cuda_graphs and pts.is_cuda and pts.shape[0] > 0:
                return self._encode_graphed(pts)
            return self._encode(pts)

    def enable_cuda_graphs(self, on=True):
        self.cuda_graphs = bool(on)
        if not on:
            self._graphs.clear()
        return self

    def _encode_graphed(self, pts):
        """CUDA-graph replay of _encode for a fixed input shape.  The graph owns its input / output / scratch buffers; the
        results are copied out, so they stay valid across later encode() calls."""
        ver = tuple((p.data_ptr(), p._version) for p in self.parameters()) + tuple((b.data_ptr(), b._version) for b in self.buffers())
        key = (tuple(pts.shape), str(pts.device), self.match_mode, self.tc_encoder)
        ent = self._graphs.get(key)
        if ent is None or ent[0] != ver:
            if len(self._graphs) >= 4:              # a handful of shapes (tracks / detections per frame); drop the oldest
                self._graphs.pop(next(iter(self._graphs)))
            static_in = pts.float().contiguous().clone()
            side = torch.cuda.Stream(device=pts.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):           # warm-up outside the capture: weight packing, kernel attributes
                self._encode(static_in)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            # thread_local: other host threads (the NCCL watchdog of a multi-rank job) may touch the CUDA API during the capture
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                static_out = self._encode(static_in)
            ent = (ver, g, static_in, static_out)
            self._graphs[key] = ent
        _, g, static_in, static_out = ent
        static_in.copy_(pts)
        g.replay()
        return static_out[0].clone(), static_out[1].clone()

    def forward_inference(self, pts_batched):
        with torch.no_grad():
            return self.backbone(pts_batched, self.backbone_list)

    def siamese_forward(self, sparse_1, sparse_2):
        assert sparse_1.shape == sparse_2.shape
        b = sparse_1.shape[0]
        with torch.no_grad():
            xyz, h = self._encode(torch.cat([sparse_1, sparse_2], dim=0))
        return xyz[:b], xyz[b:], h[:b], h[b:]

    # ------------------------------------------------------------------ pooling / heads
    def get_pooled_feats(self, h_cat):
        if self.pool_type == 'max':      # MaxPool1d over the channel axis of h.permute(0,2,1) (ReIDNet.py:527-528)
            if h_cat.shape[1] != self.output_sequence_size:
                raise NotImplementedError("pool_type='max' with channels != output_sequence_size")
            return K.cn_chanmax(_cn(h_cat))
        if self.pool_type == 'both':
            return K.cn_pool(_cn(h_cat), mode=0)
        raise NotImplementedError

    def _head_cn(self, pooled_cn):
        """match_head on channel-major pooled features (1, C, P) -> logits (P,)."""
        x = pooled_cn
        P = x.shape[2]
        # The pairs are the ROW axis here, and a pair's logit must not depend on how many other pairs share its chunk (row-sharded
        # multi-GPU driver, pair-list vs dense driver, CUDA-graph replay): ONE kernel family serves every row count of a mode.
        # Tensor-core modes: the fp32-grade 3 x tf32 TMA GEMM (pcreid_cn_linear_tma_x3; per-row sums in a fixed K order whatever the
        # row count) with the row count padded to the multiple of 4 its tensor maps need -- 0.15 -> 0.05 ms per 65 536 pairs;
        # 'parity': the FFMA kernels.  The final Linear (one output channel) is FFMA in every mode.
        x3 = self.match_mode in self.TC_MODES + ('parity_x3',) and self.head_x3 and x.is_cuda and P > 0
        if x3 and P % 4:
            x = torch.nn.functional.pad(x, (0, 4 - P % 4))
        with (K.tensor_core_linear(True, min_k=1 << 30, x3=True) if x3 else K.tensor_core_linear(False)):
            mh = self.match_head
            if (x3 and len(mh) == 2 and isinstance(mh[0], LinearRes) and mh[0].transform is None and isinstance(mh[1], nn.Linear)
                    and mh[1].out_features == 1 and mh[1].bias is not None):
                # LinearRes + Linear(C, 1): the second GroupNorm + shortcut + ReLU and the final dot in one pass (no (C, P) round trip,
                # and not a 128 x 64-tile GEMM for ONE output channel)
                pk = mh[0].packed()
                h = K.cn_groupnorm(K.cn_linear(x, pk["w1"]), pk["g1"], pk["b1"], mh[0].groups, act=K.ACT_RELU)
                h = K.cn_linear(h, pk["w2"])
                fw, fb = _final_cached(mh[1])
                return K.gn_res_relu_dot(h, pk["g2"], pk["b2"], mh[0].groups, x, fw, fb)[:P]
            for m in self.match_head:
                if isinstance(m, LinearRes):
                    x = m.forward_cn(x)
                elif isinstance(m, nn.Linear):
                    x = K.cn_linear(x, _kmajor_cached(m), bias=_bias_cached(m))
                else:
                    raise NotImplementedError(type(m))
        return x.reshape(-1)[:P]

    def xcorr_eff(self, o1, xyz1, o2, xyz2, combine='add'):
        o1__ = self.cross_stage1(o1, xyz1, o2, xyz2)
        o2__ = self.cross_stage1(o2, xyz2, o1, xyz1)
        o1 = self.cross_stage2(o1__, xyz1, o2__, xyz2)
        o2 = self.cross_stage2(o2__, xyz2, o1__, xyz1)
        if self.combine == 'add':
            out = o1 + o2
        elif self.combine == 'minus':
            out = o1 - o2
        elif self.combine == 'cat':
            out = torch.cat([o1, o2], dim=1)
        elif self.combine == 'point-cat':
            out = torch.cat([o1, o2], dim=2)
        else:
            raise NotImplementedError(self.combine)
        return out, o1, o2

    def match_forward_inference(self, h1, h2, xyz1, xyz2):
        """aligned pairs: h1/h2 (P, C, N), xyz1/xyz2 (P, N, 3) -> logits (P,)."""
        with torch.no_grad(), self._tc_match(False):
            P = h1.shape[0]
            if self.match_type == 'xcorr_eff':
                ar = torch.arange(P, device=h1.device, dtype=torch.int32)
                return self._xcorr_pairs(_cn(h1), xyz1.float().contiguous(), _cn(h2), xyz2.float().contiguous(), ar, ar)
            if self.match_type == 'concat':
                e1 = K.cn_chanmax(_cn(h1))
                e2 = K.cn_chanmax(_cn(h2))
                cat = torch.cat([e1, e2], dim=1).t().contiguous().unsqueeze(0)
                return self._head_cn(cat)
            if self.match_type in ('xcorr', 'xcorr-baseline'):
                ar = torch.arange(P, device=h1.device, dtype=torch.int32)
                return self._xcorr_search_pairs(_cn(h1), xyz1.float().contiguous(), _cn(h2), xyz2.float().contiguous(), ar, ar)
            raise NotImplementedError

    # ------------------------------------------------------------------ all-pairs driver
    def _xcorr_pairs(self, h_t, xyz_t, h_d, xyz_d, ti, dj):
        """xcorr_eff + pooling + head for the pairs (ti[p], dj[p]) -> logits (P,), fp32 parity path."""
        X1, X2 = self.cross_stage1, self.cross_stage2
        N_t, N_d = h_t.shape[2], h_d.shape[2]
        # ---- per-object work (stage 1): queries, template summaries
        q_t, q_d = X1.search_query(h_t), X1.search_query(h_d)
        wkv_t, ks_t = X1.template_summary(h_t, X1.position_code(xyz_t))
        wkv_d, ks_d = X1.template_summary(h_d, X1.position_code(xyz_d))
        pos2_t, pos2_d = X2.position_code(xyz_t), X2.position_code(xyz_d)
        # ---- per-pair work
        a = X1.attend(h_t, q_t, wkv_d, ks_d, N_d, s_map=ti, t_map=dj)       # o1__ = X1(o1 <- o2)
        b = X1.attend(h_d, q_d, wkv_t, ks_t, N_t, s_map=dj, t_map=ti)       # o2__ = X1(o2 <- o1)
        wkv_b, ks_b = X2.template_summary(b, pos2_d, pos_map=dj)
        wkv_a, ks_a = X2.template_summary(a, pos2_t, pos_map=ti)
        o1 = X2.attend(a, X2.search_query(a), wkv_b, ks_b, N_d)
        o2 = X2.attend(b, X2.search_query(b), wkv_a, ks_a, N_t)
        return self._pairs_head(o1, o2)

    def xcorr(self, search_feat, search_xyz, template_feat, template_xyz):
        """ReIDNet.xcorr (ReIDNet.py:250-256): cross -> local -> cross -> local, the search side only."""
        a = self.cross_stage1(search_feat, search_xyz, template_feat, template_xyz)
        a = self.local_stage1(a, search_xyz)
        a = self.cross_stage2(a, search_xyz, template_feat, template_xyz)
        return self.local_stage2(a, search_xyz)

    def xcorr_baseline(self, search_feat, search_xyz, template_feat, template_xyz):
        """ReIDNet.xcorr_baseline (ReIDNet.py:258-264): the two cross stages only."""
        a = self.cross_stage1(search_feat, search_xyz, template_feat, template_xyz)
        return self.cross_stage2(a, search_xyz, template_feat, template_xyz)

    def _xcorr_search_pairs(self, h_t, xyz_t, h_d, xyz_d, ti, dj):
        """'xcorr' / 'xcorr-baseline' + pooling + head for the pairs (ti[p], dj[p]): the track is the search object, the
        detection the template; BOTH cross stages attend the template's original features, so their key/value summaries
        are per-object work; only the attention read-out (and the local stages) run per pair."""
        X1, X2 = self.cross_stage1, self.cross_stage2
        N_d = h_d.shape[2]
        local = self.match_type == 'xcorr'
        wkv1, ks1 = X1.template_summary(h_d, X1.position_code(xyz_d))
        wkv2, ks2 = X2.template_summary(h_d, X2.position_code(xyz_d))
        a = X1.attend(h_t, X1.search_query(h_t), wkv1, ks1, N_d, s_map=ti, t_map=dj)
        if local:
            xyz_s = xyz_t[ti.long()].contiguous()
            a = self.local_stage1(a, xyz_s)
        a = X2.attend(a, X2.search_query(a), wkv2, ks2, N_d, t_map=dj)
        if local:
            a = self.local_stage2(a, xyz_s)
        if self.pool_type == 'both':
            return self._head_cn(K.cn_pool(a, None, mode=0, transposed=True))
        return self._head_cn(self.get_pooled_feats(a).t().contiguous().unsqueeze(0))

    def _pairs_head(self, o1, o2):
        if self.pool_type == 'both' and self.combine == 'point-cat':
            return self._head_cn(K.cn_pool(o1, o2, mode=0, transposed=True))
        out = {'add': lambda: o1 + o2, 'minus': lambda: o1 - o2, 'cat': lambda: torch.cat([o1, o2], 1),
               'point-cat': lambda: torch.cat([o1, o2], 2)}[self.combine]()
        return self._head_cn(self.get_pooled_feats(out).t().contiguous().unsqueeze(0))

    GRAPH_MAX_PAIRS = 16384     # per-frame matrices of a tracker (10 Hz replay): launch-bound sizes; scratch stays below 2 GB per graph

    def match_all_pairs(self, h_t, xyz_t, h_d, xyz_d, pair_mask=None, chunk=8192, _exact_chunk=False):
        """Dense (T, D) logit matrix; entries where ``pair_mask`` (bool (T, D), e.g. the tracker's class gate,
        tracking_point_reid.py:15-33) is False are 0, as in the reference cost matrix.
        With enable_cuda_graphs() a small dense matrix (no mask, T*D <= GRAPH_MAX_PAIRS) is replayed from a captured CUDA graph:
        its ~60 launches (per-object preparation, unit lists, fused kernels, pooling, head) cost more to issue than to run."""
        if (self.cuda_graphs and pair_mask is None and h_t.is_cuda and self.match_type != 'concat'
                and 0 < h_t.shape[0] * h_d.shape[0] <= self.GRAPH_MAX_PAIRS and self.match_mode in self.TC_MODES):
            return self._match_graphed(h_t, xyz_t, h_d, xyz_d)
        return self._match_all_pairs(h_t, xyz_t, h_d, xyz_d, pair_mask, chunk, _exact_chunk)

    def _match_graphed(self, h_t, xyz_t, h_d, xyz_d):
        """CUDA-graph replay of the dense match for fixed (T, D, N); the graph owns its inputs, scratch and output."""
        ver = tuple((p.data_ptr(), p._version) for p in self.parameters()) + tuple((b.data_ptr(), b._version) for b in self.buffers())
        key = ("match", tuple(h_t.shape), tuple(h_d.shape), str(h_t.device), self.match_mode)
        ent = self._graphs.get(key)
        if ent is None or ent[0] != ver:
            if len(self._graphs) >= 6:
                self._graphs.pop(next(iter(self._graphs)))
            static = [t.float().contiguous().clone() for t in (h_t, xyz_t, h_d, xyz_d)]
            side = torch.cuda.Stream(device=h_t.device)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):           # warm-up outside the capture: weight images, kernel attributes
                self._match_all_pairs(*static)
            torch.cuda.current_stream().wait_stream(side)
            g = torch.cuda.CUDAGraph()
            # thread_local: other host threads (the NCCL watchdog of a multi-rank job) may touch the CUDA API during the capture
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                static_out = self._match_all_pairs(*static)
            ent = (ver, g, static, static_out)
            self._graphs[key] = ent
        _, g, static, static_out = ent
        for dst, src in zip(static, (h_t, xyz_t, h_d, xyz_d)):
            dst.copy_(src)
        g.replay()
        return static_out.clone()

    def _match_all_pairs(self, h_t, xyz_t, h_d, xyz_d, pair_mask=None, chunk=8192, _exact_chunk=False):
        with torch.no_grad():
            if self.match_type == 'concat':
                return self._concat_all_pairs(_cn(h_t), _cn(h_d), pair_mask)
            ctx, chunk = self._pair_context(h_t, xyz_t, h_d, xyz_d, chunk, _exact_chunk)
            T, D = ctx[0].shape[0], ctx[2].shape[0]
            fused = ctx[4]
            out = torch.zeros((T, D), device=ctx[0].device, dtype=torch.float32)
            flat = out.view(-1)
            if pair_mask is None and fused is not None and D > 0:
                with self._tc_match(True):
                    rows_per_chunk = max(1, chunk // D)                          # dense all-pairs: whole rows per chunk
                    for r0 in range(0, T, rows_per_chunk):
                        nrows = min(rows_per_chunk, T - r0)
                        flat[r0 * D:(r0 + nrows) * D] = fused.match(ctx[5], ctx[6], None, None, dense=(r0, nrows, D))
                return out
            pairs = None if pair_mask is None else pair_mask.nonzero()
            total = T * D if pairs is None else pairs.shape[0]
            for s in range(0, total, chunk):
                e = min(total, s + chunk)
                if pairs is None:
                    lin = torch.arange(s, e, device=out.device)
                    ti, dj = lin // D, lin % D
                else:
                    ti, dj = pairs[s:e, 0], pairs[s:e, 1]
                    lin = ti * D + dj
                flat[lin] = self._pair_logits(ctx, ti, dj)
            return out

    def match_pairs(self, h_t, xyz_t, h_d, xyz_d, ti, dj, chunk=8192):
        """logits (P,) of the listed pairs (track ti[p], detection dj[p]), any order, repeats allowed: the entries
        match_all_pairs(..., pair_mask) gives those pairs.  One call serves the pairs of many scenes: a pair's logit depends on
        its two objects only.  'concat' models score through match_all_pairs (the dense pooled head)."""
        if self.match_type == 'concat':
            raise NotImplementedError("'concat' scores whole (T, D) blocks: use match_all_pairs(..., pair_mask=...)")
        with torch.no_grad():
            ctx, chunk = self._pair_context(h_t, xyz_t, h_d, xyz_d, chunk, False)
            P = ti.shape[0]
            if dj.shape[0] != P:
                raise ValueError("ti and dj must list the same number of pairs")
            out = torch.empty((P,), device=ctx[0].device, dtype=torch.float32)
            for s in range(0, P, chunk):
                e = min(P, s + chunk)
                out[s:e] = self._pair_logits(ctx, ti[s:e], dj[s:e])
            return out

    def _pair_context(self, h_t, xyz_t, h_d, xyz_d, chunk, _exact_chunk):
        """per-object work of the pair scorer -> ((h_t, xyz_t, h_d, xyz_d, fused matcher or None, packed t, packed d), chunk)"""
        h_t, h_d = _cn(h_t), _cn(h_d)
        xyz_t, xyz_d = xyz_t.float().contiguous(), xyz_d.float().contiguous()
        fused = pk_t = pk_d = None
        if self.match_mode in self.TC_MODES:
            from . import fused_pairs
            if fused_pairs.supported(self, h_t.shape[2]) and h_t.shape[2] == h_d.shape[2]:
                fused = self.fused_matcher()
                pk_t, pk_d = fused.prepare(h_t, xyz_t), fused.prepare(h_d, xyz_d)
                if not _exact_chunk:
                    chunk = max(chunk, 65536 * 256 // h_t.shape[2])
        return (h_t, xyz_t, h_d, xyz_d, fused, pk_t, pk_d), chunk

    def _pair_logits(self, ctx, ti, dj):
        """logits of one chunk of listed pairs: the one pair-list path of match_pairs and match_all_pairs"""
        h_t, xyz_t, h_d, xyz_d, fused, pk_t, pk_d = ctx
        with self._tc_match(fused is not None):
            if fused is not None:
                return fused.match(pk_t, pk_d, ti, dj)
            if self.match_type == 'xcorr_eff':
                return self._xcorr_pairs(h_t, xyz_t, h_d, xyz_d, _i32(ti), _i32(dj))
            return self._xcorr_search_pairs(h_t, xyz_t, h_d, xyz_d, _i32(ti), _i32(dj))

    def pooled_embedding(self, h):
        """'concat' match type: the per-object vector the head consumes (max over the channel axis, ReIDNet.py:455-458);
        128 floats per object -- what the row-sharded driver all-gathers instead of the per-point maps."""
        return K.cn_chanmax(_cn(h))

    def _concat_all_pairs(self, h_t, h_d, pair_mask):
        return self.concat_all_pairs_pooled(K.cn_chanmax(h_t), K.cn_chanmax(h_d), pair_mask)

    def concat_all_pairs_pooled(self, e_t, e_d, pair_mask=None):
        """'concat' head over all pairs of pooled embeddings e_t (T, E), e_d (D, E); first Linear hoisted per object
        (W1 [e_t; e_d] = W1a e_t + W1b e_d)."""
        lr, fin = self.match_head[0], self.match_head[1]
        E = e_t.shape[1]
        pk = lr.packed()
        if lr.transform is not None or pk["w1"].shape[0] != 2 * E:
            raise NotImplementedError("concat head expects LinearRes(2E, 2E)")
        w1a, w1b = _half_cached(lr, pk, E)
        A = K.cn_linear(e_t.unsqueeze(0), w1a, x1_pm=True, y_pm=True)[0]     # (T, 2E)
        Bv = K.cn_linear(e_d.unsqueeze(0), w1b, x1_pm=True, y_pm=True)[0]    # (D, 2E)
        mask = None if pair_mask is None else pair_mask.to(torch.uint8).contiguous()
        fin_w, fin_b = _final_cached(fin)          # weight vector + bias scalar, read back once per parameter version
        if self.match_mode == 'fast' and E == 128 and lr.groups * 8 == 2 * E:
            # tensor-core head (csrc/concat_tc.cu): bf16 operands for the 256 x 256 Linear, everything else fp32
            if "w2img" not in pk:
                pk["w2img"] = K.bf16_kmajor_image(lr.linear2.weight)
            return K.pair_concat_head_tc(A, Bv, e_t, e_d, pk["w2img"], pk["g1"], pk["b1"], pk["g2"], pk["b2"], fin_w, fin_b,
                                         lr.groups, mask)
        return K.pair_concat_head(A, Bv, e_t, e_d, pk["w2"], pk["g1"], pk["b1"], pk["g2"], pk["b2"], fin_w, fin_b, lr.groups, mask)

    # ------------------------------------------------------------------ mmdet BaseDetector surface
    def forward(self, return_loss=True, **kwargs):
        if return_loss:
            return self.forward_train(**kwargs)
        return self.forward_test(**kwargs)

    def forward_train(self, *args, **kwargs):
        raise NotImplementedError("pcreid_b200 implements the inference hot path; train with the reference")

    def preprocess_inputs_size_vis(self, sparse_1, sparse_2, dense_1, dense_2, label_1, label_2, id_1, id_2, size_1, size_2,
                                   vis_1, vis_2):
        st, ct = torch.stack, torch.cat
        return (st(sparse_1, 0), st(sparse_2, 0), st(dense_1, 0), st(dense_2, 0), ct(label_1, 0), ct(label_2, 0),
                ct(id_1, 0), ct(id_2, 0), ct(size_1, 0), ct(size_2, 0), ct(vis_1, 0), ct(vis_2, 0))

    def get_match_supervision(self, h1, h2, xyz1, xyz2, id_1, id_2):
        return h1, h2, xyz1, xyz2, (id_1 == id_2).float()

    def forward_test(self, sparse_1, sparse_2, dense_1, dense_2, label_1, label_2, id_1, id_2, size_1, size_2, vis_1, vis_2,
                     *args, **kwargs):
        """Same result dict as ReIDNet.forward_test (ReIDNet.py:637-689) for configs whose auxiliary heads are None."""
        (sparse_1, sparse_2, dense_1, dense_2, label_1, label_2, id_1, id_2, size_1, size_2, vis_1, vis_2) = \
            self.preprocess_inputs_size_vis(sparse_1, sparse_2, dense_1, dense_2, label_1, label_2, id_1, id_2,
                                            size_1, size_2, vis_1, vis_2)
        aux = [n for n, head in (("cls", self.cls_head), ("fp", self.fp_head), ("shape", self.shape_head))
               if head is not None and self.losses_to_use.get(n)]
        if self.losses_to_use.get("dense"):
            aux.append("dense")
        if aux:
            raise NotImplementedError(f"forward_test: the auxiliary heads / losses {aux} are built AND enabled in this config; the "
                                      "drop-in evaluates the match path (+ the kl term) only, ReIDNet.py:652-662 run the others "
                                      "-- disable them in losses_to_use or validate with the reference")
        if not self.losses_to_use.get("match", True):
            raise NotImplementedError("forward_test with losses_to_use['match']=False (ReIDNet.py:572-575 returns no predictions)")
        if self.match_type == 'concat' and self.pool_type != 'max':
            raise NotImplementedError("forward_test: the reference's match_forward pools 'concat' inputs with get_pooled_feats "
                                      "(ReIDNet.py:586-592); only pool_type='max' coincides with the channel max used here")
        xyz1, xyz2, h1, h2 = self.siamese_forward(sparse_1, sparse_2)
        h1, h2, xyz1, xyz2, match = self.get_match_supervision(h1, h2, xyz1, xyz2, id_1, id_2)
        match_preds = self.match_forward_inference(h1, h2, xyz1, xyz2)
        match_loss = self.bce(match_preds, match) * self.alpha['match']
        kl_loss = 0.
        if self.losses_to_use.get("kl"):           # get_kl_loss (ReIDNet.py:467-482): validation-only scalar over the embeddings
            lsm = torch.nn.functional.log_softmax
            kl = torch.nn.functional.kl_div(lsm(h1.reshape(h1.size(0), -1), dim=1), lsm(h2.reshape(h2.size(0), -1), dim=1),
                                            reduction='none', log_target=True).mean(dim=1)
            kl = torch.where(match == 0, -kl, kl)
            kl_loss = (kl[match == 0].mean() + kl[match == 1].mean()) * self.alpha['kl']
        zero = torch.tensor([0.])
        labels = torch.cat([label_1, label_2], dim=0)
        results = {
            'val_dense_loss': zero, 'val_fp_loss': zero, 'val_match_loss': torch.tensor([match_loss]),
            'val_shape_loss': zero, 'val_cls_loss': zero, 'val_kl_loss': torch.tensor([kl_loss]),
            'val_match_preds': match_preds, 'val_match_gt': match, 'val_cls_preds': None, 'val_cls_gt': labels,
            'val_fp_preds': None, 'val_fp_gt': (labels > 9).float(),
            'match_classes': torch.cat([label_1.unsqueeze(1), label_2.unsqueeze(1)], dim=1),
            'is_fp': torch.logical_or(label_1 > 9, label_2 > 9),
            'num_points': torch.cat([size_1.unsqueeze(1), size_2.unsqueeze(1)], dim=1),
            'val_vis_gt_all': torch.cat([vis_1.unsqueeze(1), vis_2.unsqueeze(1)], dim=1),
        }
        return [results]


# ---------------------------------------------------------------------- small caches for plain nn.Linear heads
def _cn(t):
    t = t.float()
    return t if (t.dim() == 3 and (t.stride(2) == 1 or t.shape[2] == 1)) else t.contiguous()


def _kmajor_cached(m):
    key = (m.weight.data_ptr(), m.weight._version)
    if getattr(m, "_pcreid_key", None) != key:
        m._pcreid_w = m.weight.detach().float().t().contiguous()
        m._pcreid_b = None if m.bias is None else m.bias.detach().float().contiguous()
        m._pcreid_key = key
    return m._pcreid_w


def _bias_cached(m):
    _kmajor_cached(m)
    return m._pcreid_b


def _final_cached(m):
    """final Linear(2E, 1) of the concat head: (weight vector on the device, bias as a host float).  The bias read-back is a
    device->host sync, so it happens once per parameter version instead of once per match call (and never inside a CUDA
    graph capture of the head)."""
    key = (m.weight.data_ptr(), m.weight._version, m.bias.data_ptr(), m.bias._version)
    if getattr(m, "_pcreid_fin_key", None) != key:
        m._pcreid_fin = (m.weight.detach().float().reshape(-1).contiguous(), float(m.bias.detach()[0]))
        m._pcreid_fin_key = key
    return m._pcreid_fin


def _half_cached(lr, pk, E):
    if "w1a" not in pk:
        pk["w1a"] = pk["w1"][:E].contiguous()
        pk["w1b"] = pk["w1"][E:].contiguous()
    return pk["w1a"], pk["w1b"]
