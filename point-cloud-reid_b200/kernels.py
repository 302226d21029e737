"""Thin torch-facing layer over the C ABI: allocates outputs with torch, passes raw device pointers and
the current CUDA stream.  No arithmetic happens here.

Feature tensors are channel-major ``(B, C, N)`` (the reference's layout) with unit stride along N;
arbitrary object / channel strides are passed through, so views such as ``qkv[:, :C]`` cost nothing.
"""
import ctypes
import math

import torch

from . import _lib
from . import torch_ops as _T

_OPS = _T.ops          # torch.ops.pcreid.*: one dispatcher op per compute entry point of include/pcreid.h

ACT_NONE, ACT_RELU, ACT_LEAKY02, ACT_ELU1 = 0, 1, 2, 3
TMA_TF32_MAPS, TMA_ROUND_OUT = 1, 2        # flags of pcreid_cn_linear_tma (include/pcreid.h)

# fast mode switch for cn_linear: tcgen05 kind::tf32 GEMM where the shape allows it (set by ReIDNet.set_mode / tensor_core_linear)
_TC_LINEAR = {"on": False}


class tensor_core_linear:
    """context manager: `with tensor_core_linear(True): ...` routes cn_linear through the tcgen05 kind::tf32 GEMMs.
    min_k: smallest K1 + K2 that goes to the TMA-staged kernel (pcreid_cn_linear_tma); the models pass 32 in 'fast' mode (every
    contraction with CO >= 32) and 256 in 'parity_tc' mode (the large projections only: the error budget of that mode,
    profiles/r02_parity_error_budget.md, was measured with exactly those on tf32).
    x3: contractions below min_k run on the fp32-grade 3 x tf32 variant (pcreid_cn_linear_tma_x3) instead of the FFMA kernel."""

    def __init__(self, on, min_k=None, x3=None):
        self.on, self.min_k, self.x3, self.prev = bool(on), min_k, x3, None

    def __enter__(self):
        self.prev = (_TC_LINEAR["on"], _TC_LINEAR.get("tma_min_k"), _TC_LINEAR.get("x3"))
        _TC_LINEAR["on"] = self.on
        if self.min_k is not None:
            _TC_LINEAR["tma_min_k"] = self.min_k
        if self.x3 is not None:
            _TC_LINEAR["x3"] = bool(self.x3)

    def __exit__(self, *exc):
        _TC_LINEAR["on"] = self.prev[0]
        for key, val in (("tma_min_k", self.prev[1]), ("x3", self.prev[2])):
            if val is None:
                _TC_LINEAR.pop(key, None)
            else:
                _TC_LINEAR[key] = val


def fp32_grade_only():
    """True inside the 'parity_x3' regime (every tensor-core contraction is the fp32-grade 3 x tf32 kernel): callers whose outputs feed
    a DISCRETE decision that the parity gate assumes unchanged (DGCNN's feature-space kNN) keep those contractions on the FFMA kernel,
    whose accumulation order the oracle's arithmetic was matched to."""
    return bool(_TC_LINEAR["on"] and _TC_LINEAR.get("x3") and _TC_LINEAR.get("tma_min_k", 256) >= (1 << 30))


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("pcreid_b200 kernels need CUDA tensors (there is no CPU fallback)")


def _cn(t, name):
    """validates a channel-major tensor view and returns (object stride, channel stride)."""
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32")
    if t.dim() != 3:
        raise ValueError(f"{name} must be (B, C, N)")
    if t.shape[2] > 1 and t.stride(2) != 1:
        raise ValueError(f"{name} must have unit stride along points; got strides {t.stride()}")
    return t.stride(0), t.stride(1)


def _map(m):
    if m is None:
        return None
    if m.dtype != torch.int32 or not m.is_contiguous():
        raise TypeError("object maps must be contiguous int32")
    return m


_W_IMAGES = {}


def _weight_image(w):
    """k-major (K, CO) weight -> cached tf32 operand image [(k/4)][co][k%4] for pcreid_cn_linear_tc2.  The cache holds the
    source tensor itself: its storage cannot be recycled for another weight while the entry lives, so (data_ptr, version)
    identifies it."""
    key = (w.data_ptr(), w._version, tuple(w.shape), str(w.device))
    ent = _W_IMAGES.get(key)
    if ent is None or ent[0] is not w:
        if len(_W_IMAGES) >= 256:
            _W_IMAGES.clear()
        Kd, CO = w.shape
        ent = (w, round_tf32(w).reshape(Kd // 4, 4, CO).permute(0, 2, 1).contiguous())
        _W_IMAGES[key] = ent
    return ent[1]


_W_LO = {}
# 3 x tf32 matches the FFMA kernel's error (2e-6 of the output scale) up to K = 256; the tensor core's truncating fp32 accumulation
# grows it to 8e-6 at K = 1024 (tests/test_gpu_kernels.py), too close to the 1e-4 parity gate for O(10) features: longer contractions
# stay on the FFMA kernel in the fp32-grade regime
X3_MAX_K = 256


def _lo_part(w):
    """w - hi(w), hi = the 19 bits a tcgen05 kind::tf32 MMA reads of an fp32 word (exact remainder): the second weight operand of
    pcreid_cn_linear_tma_x3.  Cached for 2-D (parameter) weights like _weight_image; per-object weights are split per call."""
    def split(t):
        return t - (t.view(torch.int32) & -8192).view(torch.float32)
    if w.dim() != 2:
        return split(w)
    key = (w.data_ptr(), w._version, tuple(w.shape), str(w.device))
    ent = _W_LO.get(key)
    if ent is None or ent[0] is not w:
        if len(_W_LO) >= 256:
            _W_LO.clear()
        ent = (w, split(w))
        _W_LO[key] = ent
    return ent[1]


def cn_linear(x1, w1, x2=None, w2=None, bias=None, act=ACT_NONE, res=None, res_after_act=False, rows=None,
              x1_map=None, x2_map=None, w1_map=None, r_map=None, x1_pm=False, x2_pm=False, out=None, B=None,
              y_pm=False):
    """Y[b,:,n] = act(W1^T X1[b,:,n] + W2^T X2[b,:,n] + bias (+res)) (+res).  w*: k-major (K, CO) or (Bw, K, CO)."""
    _need_cuda(x1, w1, x2, w2, bias, res, out)
    a = _T.linear_args()
    K1, CO = w1.shape[-2], w1.shape[-1]
    if x1_pm:
        if not x1.is_contiguous() or x1.shape[2] != K1:
            raise ValueError("point-major x1 must be contiguous (B, N, K)")
        n_in, a.x1_bs, a.ldx1 = x1.shape[1], x1.shape[1] * x1.shape[2], x1.shape[2]
    else:
        if x1.shape[1] != K1:
            raise ValueError(f"x1 has {x1.shape[1]} channels, weight expects {K1}")
        a.x1_bs, a.ldx1 = _cn(x1, "x1")
        n_in = x1.shape[2]
    rows = n_in if rows is None else rows
    if B is None:
        B = x1_map.numel() if x1_map is not None else x1.shape[0]
    a.B, a.rows, a.CO, a.K1 = B, rows, CO, K1
    a.X1, a.x1_pm, a.x1_map = x1, int(x1_pm), _map(x1_map)
    if not w1.is_contiguous() or w1.dtype != torch.float32:
        raise ValueError("weights must be contiguous float32")
    a.W1, a.w1_bs, a.w1_map = w1, (w1.shape[-2] * w1.shape[-1] if w1.dim() == 3 else 0), _map(w1_map)
    if x2 is not None:
        K2 = w2.shape[-2]
        if w2.shape[-1] != CO or not w2.is_contiguous():
            raise ValueError("w2 must be contiguous (K2, CO)")
        if x2_pm:
            if not x2.is_contiguous() or x2.shape[2] != K2:
                raise ValueError("point-major x2 must be contiguous (B, N, K)")
            a.x2_bs, a.ldx2 = x2.shape[1] * x2.shape[2], x2.shape[2]
        else:
            if x2.shape[1] != K2:
                raise ValueError(f"x2 has {x2.shape[1]} channels, weight expects {K2}")
            a.x2_bs, a.ldx2 = _cn(x2, "x2")
        a.K2, a.X2, a.x2_pm, a.x2_map = K2, x2, int(x2_pm), _map(x2_map)
        a.W2, a.w2_bs = w2, (w2.shape[-2] * w2.shape[-1] if w2.dim() == 3 else 0)
    else:
        a.K2 = 0
    a.bias = bias
    if res is not None:
        a.r_bs, a.ldr = _cn(res, "res")
        a.R, a.r_map, a.res_after_act = res, _map(r_map), int(res_after_act)
    a.act = act
    if y_pm:
        if out is None:
            out = torch.empty((B, rows, CO), device=x1.device, dtype=torch.float32)
        if not out.is_contiguous():
            raise ValueError("point-major out must be contiguous (B, rows, CO)")
        a.y_bs, a.ldy, a.y_pm = rows * CO, CO, 1
    else:
        if out is None:
            out = torch.empty((B, CO, rows), device=x1.device, dtype=torch.float32)
        a.y_bs, a.ldy = _cn(out, "out")
    a.Y = out
    # gen 3 (cn_linear_tma.cu): both operands staged by TMA tensor maps; serves every channel-major shape with CO >= 32 incl.
    # object maps and per-object weights ("tma": None = by threshold, True = always, False = never).  Below the threshold, "x3"
    # selects the fp32-grade 3 x tf32 variant of the same kernel instead of the FFMA kernel.
    tma = _TC_LINEAR.get("tma")
    if (_TC_LINEAR["on"] and tma is not False and not x1_pm and not x2_pm and not y_pm and CO >= 32 and CO % 4 == 0 and rows % 4 == 0):
        n_sms = torch.cuda.get_device_properties(x1.device).multi_processor_count
        objs = (x1.shape[0], x2.shape[0] if x2 is not None else 0, w1.shape[0] if w1.dim() == 3 else 0)
        if tma or K1 + a.K2 >= _TC_LINEAR.get("tma_min_k", 256):
            flags = ((TMA_TF32_MAPS if _TC_LINEAR.get("tma_tf32_maps", True) else 0) | (TMA_ROUND_OUT if _TC_LINEAR.get("round_out") else 0)
                     | (4 if _TC_LINEAR.get("tma_tile128") else 0))
            if _OPS.cn_linear_tma(*a.astuple(), *objs, flags, n_sms) != 3:
                return out
        elif _TC_LINEAR.get("x3") and K1 + a.K2 <= X3_MAX_K:
            if _OPS.cn_linear_tma_x3(*a.astuple(), _lo_part(w1), _lo_part(w2) if w2 is not None else None, *objs, n_sms) != 3:
                return out
    # measured on B200 (scripts/bench_linear.py): the tf32 tensor-core kernels win from K >= 256; below that the FFMA kernel
    # (up to 48 TFLOP/s) is faster
    if (_TC_LINEAR["on"] and not fp32_grade_only() and K1 + a.K2 >= _TC_LINEAR.get("min_k", 256) and x1_map is None and x2_map is None and w1_map is None
            and r_map is None and not x1_pm and not x2_pm):
        # gen 2 (warp-specialised, cn_linear_tc2.cu) wins from K >= 512: 127-141 vs 100-107 TFLOP/s on the DGCNN / PointNet heads
        if (_TC_LINEAR.get("gen", 2 if K1 + a.K2 >= 512 else 1) == 2 and w1.dim() == 2 and (w2 is None or w2.dim() == 2) and K1 % 8 == 0 and a.K2 % 8 == 0):
            n_sms = torch.cuda.get_device_properties(x1.device).multi_processor_count
            if _OPS.cn_linear_tc2(*a.astuple(), _weight_image(w1), _weight_image(w2) if w2 is not None else None, n_sms) != 3:
                return out
        if _OPS.cn_linear_tc(*a.astuple()) != 3:     # 3 == PCREID_ERR_UNSUPPORTED: shape stays on the FFMA kernel
            return out
    _OPS.cn_linear(*a.astuple())
    return out


def cn_groupnorm(x, gamma, beta, groups=1, res=None, r_map=None, act=ACT_NONE, out=None):
    """Y = act(GroupNorm_G(X) * gamma + beta (+res)) per (object, point); LayerNorm is groups=1."""
    _need_cuda(x, gamma, beta, res)
    a = _T.norm_args()
    a.B, a.C, a.rows, a.G = x.shape[0], x.shape[1], x.shape[2], groups
    a.x_bs, a.ldx = _cn(x, "x")
    a.X, a.gamma, a.beta = x, gamma, beta
    if res is not None:
        a.r_bs, a.ldr = _cn(res, "res")
        a.R, a.r_map = res, _map(r_map)
    a.act = act
    if out is None:
        out = torch.empty(tuple(x.shape), device=x.device, dtype=torch.float32)
    a.y_bs, a.ldy = _cn(out, "out")
    a.Y = out
    _OPS.cn_groupnorm(*a.astuple())
    return out


def gn_res_relu_dot(x, gamma, beta, groups, res, w, bias):
    """tail of the match head: relu(GroupNorm_G(x) * gamma + beta + res) . w + bias per column; x, res (1, C, P) channel-major,
    w (C,) on the device, bias a host float -> (P,)   (pcreid_gn_res_relu_dot)."""
    _need_cuda(x, gamma, beta, res, w)
    assert x.shape[0] == 1 and res.shape == x.shape
    _, ldx = _cn(x, "x")
    _, ldr = _cn(res, "res")
    out = torch.empty((x.shape[2],), device=x.device, dtype=torch.float32)
    _OPS.gn_res_relu_dot(x.shape[2], x.shape[1], groups, x, ldx, gamma, beta, res, ldr, w, float(bias), out)
    return out


def linattn_kv(k, v, nhead):
    """-> (Wkv (B, d, d) k-major block-diagonal, ksum (B, d)) from pre-activation keys / values (B, d, S)."""
    _need_cuda(k, v)
    B, d, S = k.shape
    k_bs, ldk = _cn(k, "k")
    v_bs, ldv = _cn(v, "v")
    wkv = torch.empty((B, d, d), device=k.device, dtype=torch.float32)
    ksum = torch.empty((B, d), device=k.device, dtype=torch.float32)
    _OPS.linattn_kv(B, S, d, nhead, k, k_bs, ldk, v, v_bs, ldv, wkv, ksum)
    return wkv, ksum


def linattn_scale(q, ksum, nhead, s_len, q_map=None, ksum_map=None, B=None):
    """Qs = (elu(q)+1) * S / ((elu(q_h)+1).ksum_h + 1e-6)."""
    _need_cuda(q, ksum)
    q_bs, ldq = _cn(q, "q")
    d, rows = q.shape[1], q.shape[2]
    if B is None:
        B = q_map.numel() if q_map is not None else (ksum_map.numel() if ksum_map is not None else q.shape[0])
    out = torch.empty((B, d, rows), device=q.device, dtype=torch.float32)
    _OPS.linattn_scale(B, rows, d, nhead, s_len, q, q_bs, ldq, _map(q_map), ksum, _map(ksum_map), out, d * rows, rows)
    return out


def local_linattn(qkv_pm, idx, nhead):
    """per-point linear attention over gathered neighbours: qkv_pm (B, N, 3C) point-major [q | k | v], idx (B, N, k) int32
    -> (B, N, C) point-major."""
    _need_cuda(qkv_pm, idx)
    if not (qkv_pm.is_contiguous() and idx.is_contiguous()) or idx.dtype != torch.int32:
        raise ValueError("local_linattn inputs must be contiguous (idx int32)")
    B, N, C3 = qkv_pm.shape
    C = C3 // 3
    out = torch.empty((B, N, C), device=qkv_pm.device, dtype=torch.float32)
    _OPS.local_linattn(B, N, C, nhead, idx.shape[2], qkv_pm, idx, out)
    return out


def cn_pool(x1, x2=None, mode=0, out=None, transposed=False):
    """mode 0: cat(max, mean) over points of x1 (and x2); mode 1: max.  -> (B, C') or, transposed, (1, C', B)."""
    _need_cuda(x1, x2)
    B, C, r1 = x1.shape
    bs1, ld1 = _cn(x1, "x1")
    bs2 = ld2 = r2 = 0
    if x2 is not None:
        bs2, ld2 = _cn(x2, "x2")
        r2 = x2.shape[2]
    Co = 2 * C if mode == 0 else C
    if out is None:
        out = torch.empty((1, Co, B) if transposed else (B, Co), device=x1.device, dtype=torch.float32)
    ob, oc = (1, B) if transposed else (Co, 1)
    _OPS.cn_pool(B, C, r1, x1, bs1, ld1, r2, x2, bs2, ld2, mode, out, ob, oc)
    return out


def cn_chanmax(x, out=None, transposed=False):
    """max over the channel axis: (B, C, N) -> (B, N) or, transposed, (1, N, B)."""
    _need_cuda(x)
    B, C, rows = x.shape
    bs, ld = _cn(x, "x")
    if out is None:
        out = torch.empty((1, rows, B) if transposed else (B, rows), device=x.device, dtype=torch.float32)
    ob, on = (1, B) if transposed else (rows, 1)
    _OPS.cn_chanmax(B, C, rows, x, bs, ld, out, ob, on)
    return out


def knn_point(k, xyz, new_xyz):
    """torch-path kNN of the backbones: int32 (B, S, k), canonical (d, idx) order."""
    _need_cuda(xyz, new_xyz)
    if not (xyz.is_contiguous() and new_xyz.is_contiguous()):
        raise ValueError("xyz / new_xyz must be contiguous")
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    idx = torch.empty((B, S, k), device=xyz.device, dtype=torch.int32)
    _OPS.knn_point(B, N, S, k, xyz, new_xyz, idx)
    return idx


def knn_point_set(k, xyz, new_xyz):
    """knn_point as an unordered set (same members, unspecified order) for consumers that max-pool over the neighbours."""
    _need_cuda(xyz, new_xyz)
    if not (xyz.is_contiguous() and new_xyz.is_contiguous()):
        raise ValueError("xyz / new_xyz must be contiguous")
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    if k > N or N > 1024 or B > 65535:
        return knn_point(k, xyz, new_xyz)
    idx = torch.empty((B, S, k), device=xyz.device, dtype=torch.int32)
    _OPS.knn_point_set(B, N, S, k, xyz, new_xyz, idx)
    return idx


def farthest_point_sample(xyz, npoint, start=None):
    """torch-path FPS of the backbones (pointnet2_utils.py:116-137): int32 (B, npoint); start (B,) = the first sample of each
    object, drawn like the reference (torch.randint on the host RNG) when not given."""
    _need_cuda(xyz)
    if not xyz.is_contiguous():
        raise ValueError("xyz must be contiguous")
    B, N, _ = xyz.shape
    if start is None:
        start = torch.randint(0, N, (B,), dtype=torch.long)
    start = start.to(device=xyz.device, dtype=torch.int32).contiguous()
    idx = torch.empty((B, npoint), device=xyz.device, dtype=torch.int32)
    _OPS.fps_torch(B, N, npoint, xyz, start, idx)
    return idx


def gather_points(features, idx):
    """features (B, C, N), idx int32 (B, M) -> (B, C, M) (pcreid_gather_points)."""
    _need_cuda(features, idx)
    features, idx = features.contiguous(), idx.contiguous()
    B, C, N = features.shape
    M = idx.shape[1]
    out = torch.empty((B, C, M), device=features.device, dtype=torch.float32)
    _OPS.gather_points(B, C, N, M, features, idx, out)
    return out


def query_ball_point(radius, nsample, xyz, new_xyz):
    """torch-path ball query of the backbones (pointnet2_utils.py:218-240): int32 (B, S, nsample), indices of the first
    nsample points with d <= radius^2 in ascending order, padded with the first."""
    _need_cuda(xyz, new_xyz)
    if not (xyz.is_contiguous() and new_xyz.is_contiguous()):
        raise ValueError("xyz / new_xyz must be contiguous")
    B, N, _ = xyz.shape
    S = new_xyz.shape[1]
    r2 = float(torch.tensor(radius ** 2, dtype=torch.float32))          # the fp32 value torch compares the distances with
    idx = torch.empty((B, S, nsample), device=xyz.device, dtype=torch.int32)
    _OPS.query_ball_point(B, N, S, r2, nsample, new_xyz, xyz, idx)
    return idx


def knn_feature(x, k):
    """DGCNN kNN in feature space: x (B, C, N) contiguous -> int32 (B, N, k)."""
    _need_cuda(x)
    B, C, N = x.shape
    x_bs, ld = _cn(x, "x")
    if C > 1 and ld != N:
        raise ValueError("x must be dense in (C, N) per object")
    idx = torch.empty((B, N, k), device=x.device, dtype=torch.int32)
    _OPS.knn_feature(B, C, N, k, x, x_bs, idx)
    return idx


def sa_edge_mlp(p1, cc, idx, w2, b2, w3, b3):
    _need_cuda(p1, cc, idx)
    B, C, N = p1.shape
    S, k = idx.shape[1], idx.shape[2]
    if not (p1.is_contiguous() and cc.is_contiguous() and idx.is_contiguous()):
        raise ValueError("sa_edge_mlp inputs must be contiguous")
    out = torch.empty((B, C, S), device=p1.device, dtype=torch.float32)
    if C > 128 or C % 16 or k > 128:
        # wider than the fused kernel's tile (mul=2 / mul=4 variants): edge tensor materialised per object chunk
        L = _lib.lib()
        step = max(1, (256 << 20) // (C * S * k * 4))
        for b0 in range(0, B, step):
            b1 = min(B, b0 + step)
            nb = b1 - b0
            h1 = torch.empty((nb, C, S * k), device=p1.device, dtype=torch.float32)
            _OPS.edge_build(nb, C, N, S, k, p1[b0:b1], cc[b0:b1], idx[b0:b1], h1)
            h3 = cn_linear(cn_linear(h1, w2, bias=b2, act=ACT_RELU), w3, bias=b3, act=ACT_RELU)
            _OPS.seg_max(nb * C * S, k, h3, out[b0:b1])
        return out
    _OPS.sa_edge_mlp(B, C, N, S, k, p1, cc, idx, w2, b2, w3, b3, out)
    return out


def round_tf32(w):
    """fp32 -> nearest tf32 value (ties away from zero), kept in fp32 storage.  tcgen05 kind::tf32 ignores the low 13 mantissa
    bits of its operands (truncation); weights that are pre-rounded here carry half the error and no bias towards zero."""
    bits = w.detach().float().contiguous().view(torch.int32)
    return ((bits + 0x1000) & ~0x1fff).view(torch.float32)


def tf32_image(w):
    """(C_out, C_in) fp32 weight -> tcgen05 K-major operand image [k/4][n][4] (tf32-rounded values in fp32 storage)."""
    n, kd = w.shape
    return round_tf32(w).reshape(n, kd // 4, 4).permute(1, 0, 2).contiguous()


def tf32_image_padded(w, k_pad):
    """tf32_image of a (C_out, C_in) weight whose input channels are zero-padded to k_pad."""
    w = w.detach().float()
    if w.shape[1] < k_pad:
        w = torch.cat([w, w.new_zeros(w.shape[0], k_pad - w.shape[1])], 1)
    return tf32_image(w)


def weight_blob(*images):
    """concatenation of operand images in the order a fused kernel consumes them (attn_tc.cu)."""
    return torch.cat([i.reshape(-1) for i in images]).contiguous()


def attn_front(xyz, feat, wp0, bp0, bp2, blob, DP, NFP, NF):
    """key-side half of a linear-attention block on the tensor cores: pos MLP, feat + pos, projections.
    -> (B, NFP + NF, S): the first NFP channels are projections of feat + pos, the rest of feat."""
    _need_cuda(xyz, feat, blob)
    B, C2, S = feat.shape
    f_bs, ldf = _cn(feat, "feat")
    if not xyz.is_contiguous():
        raise ValueError("xyz must be contiguous")
    L = _lib.lib()
    if blob.numel() * 4 != L.pcreid_attn_front_blob_bytes(C2, DP, NFP, NF):
        raise ValueError("attn_front: weight blob does not match the shapes")
    out = torch.empty((B, NFP + NF, S), device=feat.device, dtype=torch.float32)
    _OPS.attn_front(B, S, C2, DP, NFP, NF, xyz, feat, f_bs, ldf, wp0, bp0, bp2, blob, out, out.stride(0), out.stride(1))
    return out


def linattn_kv_img(k, v, nhead, rows_q):
    """KV summaries of linear attention as per-object, per-head tcgen05 operand images + Ksum, from pre-activation keys /
    values (B, d, S) channel-major views.  rows_q = query rows per object of the attn_back call that will consume them
    (objects of a packed tile must be contiguous, so the allocation is rounded up to the tile's object count)."""
    _need_cuda(k, v)
    B, d, S = k.shape
    k_bs, ldk = _cn(k, "k")
    v_bs, ldv = _cn(v, "v")
    L = _lib.lib()
    opt = L.pcreid_attn_back_objects_per_tile(rows_q, d)
    kvimg = torch.empty(((B + opt - 1) // opt * opt, d * (d // nhead)), device=k.device, dtype=torch.float32)
    ksum = torch.empty((B, d), device=k.device, dtype=torch.float32)
    _OPS.linattn_kv_img(B, S, d, nhead, k, k_bs, ldk, v, v_bs, ldv, kvimg, ksum)
    return kvimg, ksum


def attn_back(feat1, q, ksum, kvimg, g1, b1, g2, b2, blob, nhead, CO, residual, feat1_pm=False):
    """query-side half of a linear-attention block: (q | Wq feat1) -> elu+1 -> . KV per head -> / (Q.Ksum) -> merge -> LN1
    -> mlp -> LN2 (+ feat1)."""
    _need_cuda(feat1, q, ksum, kvimg, blob)
    D = ksum.shape[1]
    if feat1_pm:
        if not feat1.is_contiguous():
            raise ValueError("point-major feat1 must be contiguous (B, rows, C1)")
        B, rows, C1 = feat1.shape
        f1_bs, ldf1 = rows * C1, C1
    else:
        B, C1, rows = feat1.shape
        f1_bs, ldf1 = _cn(feat1, "feat1")
    q_bs = ldq = 0
    if q is not None:
        q_bs, ldq = _cn(q, "q")
    L = _lib.lib()
    if blob.numel() * 4 != L.pcreid_attn_back_blob_bytes(D, (C1 + 7) // 8 * 8, CO, int(q is not None)):
        raise ValueError("attn_back: weight blob does not match the shapes")
    opt = L.pcreid_attn_back_objects_per_tile(rows, D)
    if kvimg.shape[0] < (B + opt - 1) // opt * opt:
        raise ValueError("attn_back: kvimg must hold the objects of the last tile (use linattn_kv_img(..., rows_q=rows))")
    out = torch.empty((B, CO, rows), device=feat1.device, dtype=torch.float32)
    _OPS.attn_back(B, rows, D, nhead, C1, CO, int(residual), int(feat1_pm), feat1, f1_bs, ldf1, q, q_bs, ldq, ksum, kvimg, g1, b1, g2, b2, blob, out, out.stride(0), out.stride(1))
    return out


def sa_edge_mlp_tc(p1, cc, idx, w2img, b2, w3img, b3, gen=2):
    """tensor-core (tf32) version of sa_edge_mlp; w*img from tf32_image(); p1 (B, N, C) and cc (B, S, C) point-major.
    gen=2: warp-specialised kernel with both A operands in tensor memory (sa_tc2.cu); shapes it does not cover (k < 16)
    and gen=1 run the first-generation kernel (sa_tc.cu)."""
    _need_cuda(p1, cc, idx)
    B, N, C = p1.shape
    S, k = idx.shape[1], idx.shape[2]
    if not (p1.is_contiguous() and cc.is_contiguous() and idx.is_contiguous()):
        raise ValueError("sa_edge_mlp_tc inputs must be contiguous")
    out = torch.empty((B, C, S), device=p1.device, dtype=torch.float32)
    n_sms = torch.cuda.get_device_properties(p1.device).multi_processor_count
    if gen == 2:
        if _OPS.sa_edge_mlp_tc2(B, C, N, S, k, p1, cc, idx, w2img, b2, w3img, b3, out, 0, n_sms) != 3:
            return out
    _OPS.sa_edge_mlp_tc(B, C, N, S, k, p1, cc, idx, w2img, b2, w3img, b3, out, n_sms)
    return out


def edge_gather_max(p, q, idx, act, out=None):
    _need_cuda(p, q, idx)
    B, C, N = p.shape
    k = idx.shape[2]
    if not (p.is_contiguous() and q.is_contiguous() and idx.is_contiguous()):
        raise ValueError("edge_gather_max inputs must be contiguous")
    if out is None:
        out = torch.empty((B, C, N), device=p.device, dtype=torch.float32)
    o_bs, ldo = _cn(out, "out")
    _OPS.edge_gather_max(B, C, N, k, p, q, idx, act, out, o_bs, ldo)
    return out


def pair_concat_head(a, bv, et, ed, w2, g1, be1, g2, be2, w, b0, groups, mask=None):
    _need_cuda(a, bv, et, ed)
    T, D, E = a.shape[0], bv.shape[0], et.shape[1]
    out = torch.empty((T, D), device=a.device, dtype=torch.float32)
    _OPS.pair_concat_head(T, D, E, groups, a, bv, et, ed, w2, g1, be1, g2, be2, w, float(b0), mask, out)
    return out


LSAP_MAX_SIZE, LSAP_MAX_BATCH = 4096, 65535


def linear_assignment(score, min_score, pair_mask=None):
    """Maximum-weight matching of tracks to detections (pcreid_lsap).  score (T, D) or (B, T, D) CUDA float32, higher = more
    alike (the logits of match_all_pairs); pair_mask bool of the same shape or None (e.g. class_gate).  A pair may be matched
    only when pair_mask allows it, its score is finite and score > min_score; the matching maximises the sum of
    score - min_score (float64).  -> (det_for_track (..., T), track_for_det (..., D)) int64 on the device, -1 = unmatched.
    Checks shapes only: no host synchronisation, so the call can be captured in a CUDA graph."""
    _need_cuda(score, pair_mask)
    if score.dtype != torch.float32:
        raise TypeError("score must be float32")
    if score.dim() not in (2, 3):
        raise ValueError(f"score must be (T, D) or (B, T, D); got {tuple(score.shape)}")
    if isinstance(min_score, torch.Tensor):
        raise TypeError("min_score must be a Python number (reading a tensor would synchronise)")
    tau = float(min_score)
    if not math.isfinite(tau):
        raise ValueError("min_score must be finite")
    batched = score.dim() == 3
    s = score if batched else score.unsqueeze(0)
    B, T, D = s.shape
    if T > LSAP_MAX_SIZE or D > LSAP_MAX_SIZE or B > LSAP_MAX_BATCH:
        raise ValueError(f"linear_assignment supports T, D <= {LSAP_MAX_SIZE} and B <= {LSAP_MAX_BATCH}; got {(B, T, D)}")
    mask = None
    if pair_mask is not None:
        if pair_mask.dtype != torch.bool or pair_mask.shape != score.shape:
            raise ValueError("pair_mask must be a bool tensor of the score's shape")
        if pair_mask.device != score.device:
            raise ValueError("pair_mask must be on the score's device")
        mask = (pair_mask if batched else pair_mask.unsqueeze(0)).contiguous()
    s = s.contiguous()
    det_for_track = torch.empty((B, T), device=s.device, dtype=torch.int32)
    track_for_det = torch.empty((B, D), device=s.device, dtype=torch.int32)
    work = torch.empty((B * _lib.lib().pcreid_lsap_workspace_bytes(T, D),), device=s.device, dtype=torch.uint8)
    _OPS.lsap(B, T, D, s, mask, tau, det_for_track, track_for_det, work)
    det_for_track, track_for_det = det_for_track.long(), track_for_det.long()
    if not batched:
        return det_for_track[0], track_for_det[0]
    return det_for_track, track_for_det


def linear_assignment_blocks(score, shapes, min_score, pair_mask=None):
    """linear_assignment over B problems of different shapes in one launch (pcreid_lsap_blocks), e.g. one per scene.
    score: 1-D CUDA float32 of sum T_b * D_b, problem b's row-major (T_b, D_b) block after problem b-1's; shapes: host sequence
    of (T_b, D_b); pair_mask: bool, packed like score, or None.  Each problem's result equals linear_assignment on its block.
    -> packed int64 (det_for_track (sum T_b,), track_for_det (sum D_b,)) on the device, -1 = unmatched.  Validates the shapes on
    the host and never reads device memory back (no host synchronisation)."""
    _need_cuda(score, pair_mask)
    if score.dtype != torch.float32 or score.dim() != 1:
        raise TypeError("score must be 1-D float32 (problems packed one after another)")
    if isinstance(min_score, torch.Tensor):
        raise TypeError("min_score must be a Python number (reading a tensor would synchronise)")
    tau = float(min_score)
    if not math.isfinite(tau):
        raise ValueError("min_score must be finite")
    shapes = [(int(t), int(d)) for t, d in shapes]
    B = len(shapes)
    if B > LSAP_MAX_BATCH or any(t < 0 or d < 0 or t > LSAP_MAX_SIZE or d > LSAP_MAX_SIZE for t, d in shapes):
        raise ValueError(f"linear_assignment_blocks supports 0 <= T, D <= {LSAP_MAX_SIZE} and at most {LSAP_MAX_BATCH} problems")
    L = _lib.lib()
    offs = [[0] for _ in range(4)]
    for t, d in shapes:
        for row, v in zip(offs, (t, d, t * d, L.pcreid_lsap_workspace_bytes(t, d))):
            row.append(row[-1] + v)
    if score.numel() != offs[2][-1]:
        raise ValueError(f"score holds {score.numel()} elements; the shapes need {offs[2][-1]}")
    if pair_mask is not None:
        if pair_mask.dtype != torch.bool or pair_mask.shape != score.shape:
            raise ValueError("pair_mask must be a bool tensor of the score's shape")
        if pair_mask.device != score.device:
            raise ValueError("pair_mask must be on the score's device")
        pair_mask = pair_mask.contiguous()
    dev = score.device
    det_for_track = torch.empty((offs[0][-1],), device=dev, dtype=torch.int32)
    track_for_det = torch.empty((offs[1][-1],), device=dev, dtype=torch.int32)
    work = torch.empty((offs[3][-1],), device=dev, dtype=torch.uint8)
    off = torch.tensor(offs, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)
    _OPS.lsap_blocks(B, max((t for t, _ in shapes), default=0), max((d for _, d in shapes), default=0), off, score.contiguous(),
                     pair_mask, tau, det_for_track, track_for_det, work)
    return det_for_track.long(), track_for_det.long()


TRACK_MAX_CAPACITY, TRACK_MAX_SCENES = 4096, 65535
# the device state of a track table (models/tracking.py, TrackTable): (attribute, dtype, trailing shape); per slot (S, C, ...),
# per scene (S,)
TRACK_SLOT_FIELDS = (("alive", torch.bool, ()), ("track_id", torch.int64, ()), ("label", torch.int32, ()),
                     ("length", torch.int32, ()), ("age", torch.int32, ()), ("hits", torch.int32, ()),
                     ("box", torch.float32, (7,)), ("active", torch.int32, ()))
TRACK_SCENE_FIELDS = (("next_id", torch.int64), ("dropped", torch.int64), ("count", torch.int32))


def _track_state(table):
    """checks the table's tensors (pcreid_track_* layout) on the host -> (S, C, device)"""
    S, C = table.alive.shape
    if C < 1 or C > TRACK_MAX_CAPACITY or S > TRACK_MAX_SCENES:
        raise ValueError(f"track tables support 1 <= capacity <= {TRACK_MAX_CAPACITY} and at most {TRACK_MAX_SCENES} scenes")
    dev = table.alive.device
    _need_cuda(table.alive)
    for name, dtype, tail in TRACK_SLOT_FIELDS:
        t = getattr(table, name)
        if t.dtype != dtype or tuple(t.shape) != (S, C) + tail or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"table.{name} must be contiguous {dtype} of shape {(S, C) + tail} on {dev}")
    for name, dtype in TRACK_SCENE_FIELDS:
        t = getattr(table, name)
        if t.dtype != dtype or tuple(t.shape) != (S,) or t.device != dev:
            raise ValueError(f"table.{name} must be {dtype} of shape {(S,)} on {dev}")
    return S, C, dev


def _track_offsets(shapes, S, C, dev):
    """host (A_s, D_s) per scene -> (shapes, host prefix sums [3][S + 1], the same on the device through pinned memory)"""
    shapes = [(int(a), int(d)) for a, d in shapes]
    if len(shapes) != S:
        raise ValueError(f"{len(shapes)} block shapes for {S} scenes")
    if any(a < 0 or d < 0 or a > C or d > TRACK_MAX_CAPACITY for a, d in shapes):
        raise ValueError(f"every scene needs 0 <= A_s <= capacity ({C}) and 0 <= D_s <= {TRACK_MAX_CAPACITY}")
    offs = [[0] for _ in range(3)]
    for a, d in shapes:
        for row, v in zip(offs, (a, d, a * d)):
            row.append(row[-1] + v)
    return shapes, offs, torch.tensor(offs, dtype=torch.int64).pin_memory().to(dev, non_blocking=True)


def _det_arrays(n, det_label, det_length, det_box, dev):
    for name, t, dtype, shape in (("det_label", det_label, torch.int32, (n,)), ("det_length", det_length, torch.int32, (n,)),
                                  ("det_box", det_box, torch.float32, (n, 7))):
        if t.dtype != dtype or tuple(t.shape) != shape or t.device != dev:
            raise ValueError(f"{name} must be {dtype} of shape {shape} on {dev}")
    return det_label.contiguous(), det_length.contiguous(), det_box.contiguous()


def track_gate_blocks(table, shapes, det_label, det_length, det_box, num_classes=8, min_points=2, use_lengths=True,
                      radius_sq=None):
    """Packed class gate of every scene's (A_s, D_s) block (pcreid_track_gate_blocks).  table: the device state of a track
    table (TRACK_SLOT_FIELDS / TRACK_SCENE_FIELDS, e.g. models/tracking.py TrackTable); shapes: host (A_s, D_s) per scene,
    A_s = active tracks (0 for a scene without a frame); det_label / det_length int32 (sum D_s,), det_box f32 (sum D_s, 7)
    packed over the scenes; radius_sq: None or f32 (num_classes,) squared ground-plane radius per class on the device.
    -> bool (sum A_s * D_s,), scene s's row-major block after scene s-1's (the packing linear_assignment_blocks reads).
    Checks shapes on the host and never reads device memory back."""
    S, C, dev = _track_state(table)
    shapes, offs, off = _track_offsets(shapes, S, C, dev)
    det_label, det_length, det_box = _det_arrays(offs[1][-1], det_label, det_length, det_box, dev)
    if radius_sq is not None and (radius_sq.dtype != torch.float32 or tuple(radius_sq.shape) != (num_classes,)
                                  or radius_sq.device != dev):
        raise ValueError(f"radius_sq must be float32 of shape ({num_classes},) on {dev}")
    gate = torch.empty((offs[2][-1],), device=dev, dtype=torch.bool)
    _OPS.track_gate_blocks(S, C, max((a for a, _ in shapes), default=0), max((d for _, d in shapes), default=0), off,
                           table.active, table.label, table.length, table.box, det_label, det_length, det_box,
                           int(num_classes), int(min_points), int(bool(use_lengths)),
                           None if radius_sq is None else radius_sq.contiguous(), gate)
    return gate


def track_update(table, shapes, track_for_det, det_label, det_length, det_box, max_age=None, replace_all=False):
    """One step of the track table's bookkeeping for every scene in one launch (pcreid_track_update): matched tracks, ageing and
    retirement past max_age (None: never), unmatched detections into the lowest free slots, the next active lists and counts.
    shapes / det_*: as track_gate_blocks; track_for_det int64 (sum D_s,): position in the scene's active list or -1 (the output
    of linear_assignment_blocks on the gate).  Updates table in place -> (det_track_id int64 (sum D_s,), -1 for a dropped
    detection; det_row int32 (sum D_s,): the global table row that receives the detection's observation, -1 if none).
    Checks shapes on the host and never reads device memory back."""
    S, C, dev = _track_state(table)
    shapes, offs, off = _track_offsets(shapes, S, C, dev)
    n = offs[1][-1]
    det_label, det_length, det_box = _det_arrays(n, det_label, det_length, det_box, dev)
    if track_for_det.dtype != torch.int64 or tuple(track_for_det.shape) != (n,) or track_for_det.device != dev:
        raise ValueError(f"track_for_det must be int64 of shape ({n},) on {dev}")
    if max_age is not None and int(max_age) < 0:
        raise ValueError("max_age must be None or >= 0")
    det_track_id = torch.empty((n,), device=dev, dtype=torch.int64)
    det_row = torch.empty((n,), device=dev, dtype=torch.int32)
    _OPS.track_update(S, C, max((d for _, d in shapes), default=0), off, track_for_det.contiguous(), det_label, det_length,
                      det_box, -1 if max_age is None else int(max_age), int(bool(replace_all)), table.alive,
                      table.track_id, table.label, table.length, table.age, table.hits, table.box, table.next_id,
                      table.dropped, table.active, table.count, det_track_id, det_row)
    return det_track_id, det_row


# the motion state of a track table built with motion (models/tracking.py, MotionModel): the constant-velocity Kalman filter's
# box estimate, velocity and compact covariance per slot (layout: include/pcreid.h, pcreid_track_predict)
TRACK_MOTION_FIELDS = (("kf_box", torch.float32, (7,)), ("kf_vel", torch.float32, (3,)), ("kf_cov", torch.float32, (13,)))


def _track_motion_state(table, S, C, dev):
    for name, dtype, tail in TRACK_MOTION_FIELDS:
        t = getattr(table, name, None)
        if t is None or t.dtype != dtype or tuple(t.shape) != (S, C) + tail or not t.is_contiguous() or t.device != dev:
            raise ValueError(f"table.{name} must be contiguous {dtype} of shape {(S, C) + tail} on {dev} (a table with motion)")


def _finite_scalars(**kw):
    for name, (v, positive) in kw.items():
        if isinstance(v, torch.Tensor):
            raise TypeError(f"{name} must be a Python number (reading a tensor would synchronise)")
        v = float(v)
        if not math.isfinite(v) or v < 0 or (positive and v == 0):
            raise ValueError(f"{name} must be finite and {'> 0' if positive else '>= 0'}; got {v}")


def track_dt(dt, S, frozen=()):
    """a float or one value per scene -> S floats, each finite and >= 0; the entries of the scenes listed in frozen (which
    are not predicted) are not read and become 0.0"""
    try:
        dt = list(dt)
    except TypeError:
        dt = [dt] * S
    if len(dt) != S:
        raise ValueError(f"{len(dt)} dt values for {S} scenes")
    frozen = set(frozen)
    dt = [0.0 if s in frozen else v for s, v in enumerate(dt)]
    _finite_scalars(**{f"dt[{s}]": (v, False) for s, v in enumerate(dt)})
    return [float(v) for v in dt]


def track_predict(table, shapes, dt, q=1.0, q_vel=0.01):
    """Kalman prediction of every active track of every scene in one launch (pcreid_track_predict): box += dt * velocity and
    the covariance grows by the process noise q (box values) / q_vel (velocity).  shapes: host (A_s, D_s) per scene as
    track_gate_blocks (a scene without a frame has A_s = 0 and is not predicted); dt: host float or one per scene, each finite
    and >= 0, sent as float32 through pinned memory.  Updates table.kf_box / kf_vel / kf_cov in place.  Checks on the host and
    never reads device memory back."""
    S, C, dev = _track_state(table)
    _track_motion_state(table, S, C, dev)
    shapes, offs, off = _track_offsets(shapes, S, C, dev)
    _finite_scalars(q=(q, False), q_vel=(q_vel, False))
    dt = torch.tensor(track_dt(dt, S), dtype=torch.float32).pin_memory().to(dev, non_blocking=True)
    _OPS.track_predict(S, C, max((a for a, _ in shapes), default=0), off, table.active, dt, table.kf_box, table.kf_vel,
                       table.kf_cov, float(q), float(q_vel))


def track_correct(table, shapes, track_rows, track_for_det, det_box, det_row, init_var=10.0, init_vel_var=1e4, r=1.0):
    """Kalman correction after track_update of the same step, every scene in one launch (pcreid_track_correct): a matched
    detection corrects its track with its box (measurement noise r; yaw with AB3DMOT's flipped-heading rule), an unmatched one
    that received a slot starts that slot's filter (box, velocity 0, covariance init_var / init_vel_var); a dropped one changes
    nothing.  shapes / det_box: as track_update; track_rows int64 (sum A_s,): the active rows entering the step, packed by scene
    (table.active before track_update); track_for_det int64 and det_row int32 (sum D_s,): the inputs and the output of
    track_update.  Updates table.kf_box / kf_vel / kf_cov in place.  Checks on the host and never reads device memory back."""
    S, C, dev = _track_state(table)
    _track_motion_state(table, S, C, dev)
    shapes, offs, off = _track_offsets(shapes, S, C, dev)
    _finite_scalars(init_var=(init_var, True), init_vel_var=(init_vel_var, True), r=(r, True))
    n = offs[1][-1]
    for name, t, dtype, shape in (("track_rows", track_rows, torch.int64, (offs[0][-1],)),
                                  ("track_for_det", track_for_det, torch.int64, (n,)),
                                  ("det_box", det_box, torch.float32, (n, 7)), ("det_row", det_row, torch.int32, (n,))):
        if t.dtype != dtype or tuple(t.shape) != shape or t.device != dev:
            raise ValueError(f"{name} must be {dtype} of shape {shape} on {dev}")
    _OPS.track_correct(S, C, max((d for _, d in shapes), default=0), off, track_rows.contiguous() if track_rows.numel() else None,
                       track_for_det.contiguous(), det_box.contiguous(), det_row.contiguous(), table.kf_box, table.kf_vel,
                       table.kf_cov, float(init_var), float(init_vel_var), float(r))


def track_gate_motion_blocks(table, shapes, det_label, det_length, det_box, num_classes=8, min_points=2, use_lengths=True,
                             radius_sq=None, r=1.0, gate_chi2=None):
    """track_gate_blocks on the predicted boxes (table.kf_box, after track_predict) of a table with motion
    (pcreid_track_gate_motion_blocks): class_gate's rule, radius_sq around the predicted centre, and when gate_chi2 is given
    fl(dx*dx / Sx + dy*dy / Sy) <= gate_chi2 with Sx, Sy = the x / y position variance + r (the Mahalanobis distance of the
    ground-plane innovation).  -> bool (sum A_s * D_s,) packed as track_gate_blocks.  Checks on the host and never reads device
    memory back."""
    S, C, dev = _track_state(table)
    _track_motion_state(table, S, C, dev)
    shapes, offs, off = _track_offsets(shapes, S, C, dev)
    det_label, det_length, det_box = _det_arrays(offs[1][-1], det_label, det_length, det_box, dev)
    if radius_sq is not None and (radius_sq.dtype != torch.float32 or tuple(radius_sq.shape) != (num_classes,)
                                  or radius_sq.device != dev):
        raise ValueError(f"radius_sq must be float32 of shape ({num_classes},) on {dev}")
    _finite_scalars(r=(r, True))
    if gate_chi2 is not None:
        _finite_scalars(gate_chi2=(gate_chi2, True))
    gate = torch.empty((offs[2][-1],), device=dev, dtype=torch.bool)
    _OPS.track_gate_motion_blocks(S, C, max((a for a, _ in shapes), default=0), max((d for _, d in shapes), default=0), off,
                                  table.active, table.label, table.length, table.kf_box, det_label, det_length, det_box,
                                  int(num_classes), int(min_points), int(bool(use_lengths)),
                                  None if radius_sq is None else radius_sq.contiguous(), table.kf_cov, float(r),
                                  0.0 if gate_chi2 is None else float(gate_chi2), gate)
    return gate


def _rows(src, dst, name):
    """(n, ...) source rows and (R, ...) table rows of one dtype and row shape -> bytes per row"""
    if src.dtype != dst.dtype or src.shape[1:] != dst.shape[1:] or src.device != dst.device or not dst.is_contiguous():
        raise ValueError(f"{name}: rows of {tuple(src.shape[1:])} {src.dtype} into a contiguous table of "
                         f"{tuple(dst.shape[1:])} {dst.dtype}")
    return math.prod(dst.shape[1:]) * dst.element_size()


def track_scatter(det_row, det_xyz, det_feat, xyz, feat):
    """xyz[det_row[d]] = det_xyz[d] and feat[det_row[d]] = det_feat[d] for every d with det_row[d] >= 0, in one launch
    (pcreid_track_scatter); rows are copied as bytes, so any dtype works.  det_row int32 (n,) from track_update."""
    _need_cuda(det_row, det_xyz, det_feat, xyz, feat)
    n = det_row.shape[0]
    if det_row.dtype != torch.int32 or det_row.dim() != 1 or det_xyz.shape[0] != n or det_feat.shape[0] != n:
        raise ValueError("det_row must be int32 (n,) with one xyz and one feature row per entry")
    bx, bf = _rows(det_xyz, xyz, "xyz"), _rows(det_feat, feat, "feat")
    _OPS.track_scatter(n, det_row.contiguous(), bx, det_xyz.contiguous(), xyz, bf, det_feat.contiguous(), feat)


def bf16_kmajor_image(w):
    """torch weight (N, K) -> bf16 K-major tcgen05 operand image [K/8][N][8] (uint8 view)."""
    n, kd = w.shape
    return w.detach().to(torch.bfloat16).view(n, kd // 8, 8).permute(1, 0, 2).contiguous().view(torch.uint8).flatten()


def pair_concat_head_tc(a, bv, et, ed, w2img, g1, be1, g2, be2, w, b0, groups, mask=None):
    """tensor-core version of pair_concat_head (bf16 operands for the 256 x 256 Linear, fp32 GroupNorms / accumulation)."""
    _need_cuda(a, bv, et, ed, w2img)
    T, D, E = a.shape[0], bv.shape[0], et.shape[1]
    out = torch.empty((T, D), device=a.device, dtype=torch.float32)
    n_ctas = torch.cuda.get_device_properties(a.device).multi_processor_count
    _OPS.pair_concat_head_tc(T, D, E, groups, a, bv, et, ed, w2img, g1, be1, g2, be2, w, float(b0), mask, out, n_ctas)
    return out
