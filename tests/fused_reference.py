"""Float64 restatement of the fused tensor-core `xcorr_eff` matcher, one function per kernel of the chain
(csrc/pair_tc.cu, csrc/pair_tc2.cu, host side models/fused_pairs.py):

    pack / pack_bias / pack_b7 -> phase1a (pair_p1a2) -> phase1b (pair_p1b_n) -> phase2 (pair_p2y) -> pool_finish (pool_finish2)

It restates the contract of include/pcreid.h (section B') rather than the kernels' code: every GEMM is an exact float64 product of
the decoded 16-bit operands, every LayerNorm and attention normalisation is exact, and the result is rounded to the operand format
(`fmt`: FMT_BF16 'fast', FMT_F16 'parity_tc') exactly where a kernel stores a 16-bit operand:

  * pack:    the per-object images QF1 = elu(Wq1 h) + 1, H = h + beta2, PV = Wv2 pos2(xyz), the attention operand MK1;
  * phase1a: X' (LayerNorm1 output), the ReLU hidden layer, the stage-1 output A;
  * phase1b: the key / value operands Kf, V of the key/value product, blockdiag(KV), the stage-2 operand B7;
  * phase2:  the queries Qf, X', the ReLU hidden layer (the stage-2 output o - beta2 stays fp32 and is pooled).

fp16 conversions saturate to +-65504 (cvt.rn.satfinite); bf16 conversions round to nearest even.

Deliberate approximations of the kernels that are part of their documented arithmetic, mirrored here and therefore NOT counted
as errors by the tests:
  * the stage-2 query feature is computed as max(x', 0) c + 2^min(x', 0) from x' = (Wq / c) a with c = LN2B = bf16(ln 2) in the
    bf16 kernels and c = ln 2 in the fp16 ones (tc_common.cuh elu1_scaled); in bf16 that is exp(x ln2 / LN2B) = exp(1.0028 x)
    for negative x instead of exp(x);
  * the bf16 kernels evaluate elu(k) + 1 of the keys on packed bf16 pairs: k is rounded to bf16, multiplied by bf16(log2 e) =
    1.4453125 (rounded again), raised to 2^ (rounded) and added (rounded); the value operand is v rounded to bf16 plus the PV
    image, rounded again (tc_common.cuh bf2_elu1, OpBF16::add).  The fp16 kernels do the same in fp32 and round once.
Not mirrored: ex2.approx / __expf / rsqrtf are approximate (a few fp32 ulps), and accumulation is fp32 instead of float64.  Both are
far below one 16-bit ulp; where they tip a rounding of an intermediate operand the difference is one ulp of that operand, which
is what the tests' tolerances allow for.

LayerNorm inputs are taken as centred (no mean subtraction), as the kernels do: the host centres the merge and mlp[2] weights
over their output channels, so the mean is zero by construction (a broken centring must show up as an error, not be absorbed).
Activations are point-major here: (..., points, 64 channels).
"""
import math

import torch
import torch.nn.functional as F

FMT_BF16, FMT_F16 = 0, 1
ACT_NONE, ACT_ELU1 = 0, 3          # PCREID_ACT_NONE / PCREID_ACT_ELU1
LN_EPS = 1e-5                # LayerNorm eps (pair_common.cuh LN_EPS)
ATT_EPS = 1e-6               # LinearAttention.eps
F16_MAX = 65504.0
LN2B = 0.69140625            # bf16(ln 2)
LOG2E_B = 1.4453125          # bf16(log2 e): the multiplier of the packed bf16 elu
UNIT_ROUNDOFF = {FMT_F16: 2.0 ** -11, FMT_BF16: 2.0 ** -8}
DTYPE = {FMT_F16: torch.float16, FMT_BF16: torch.bfloat16}
D = 64                       # d_model of the fused matcher (2 heads of 32)

# weight blob layouts (bytes): pair_tc2.cu Q1A_* / Q2_*, pair_tc.cu P1B_*
_W0EXT_BYTES = 128 * 144 * 2
_W2_BYTES = 64 * 128 * 2
_W64_BYTES = 64 * 64 * 2


def to_fmt(x, fmt):
    """round to the 16-bit operand format (round to nearest even; fp16 saturates), returned as float64"""
    x = x.double()
    if fmt == FMT_F16:
        x = x.clamp(-F16_MAX, F16_MAX)
    return x.to(DTYPE[fmt]).double()


def elu1(x):
    return F.elu(x) + 1.0


def pack(x, fmt, act=ACT_NONE, bias=None):
    """pcreid_pack_image / pcreid_pack_image_bias of one element each: fmt(x + bias) or fmt(elu(x) + 1).  x + bias is formed in
    fp32 (the kernel's one fp32 add), so that the bias packer can be checked bit for bit."""
    if bias is not None:
        x = (x.float() + bias.float()).double()
    x = x.double()
    if act == ACT_ELU1:
        x = elu1(x)
    return to_fmt(x, fmt)


def pack_b7(M, ksum, fmt):
    """pcreid_pack_b7: M (..., 64 d, 64 out) fp32 + ksum (..., 64) -> attention operand (..., 2 heads, 32 k, 80 n):
    n < 64 the merged output channels M[32 h + k, n], n = 64 Ksum[32 h + k], n > 64 zero"""
    out = torch.zeros(*M.shape[:-2], 2, 32, 80, dtype=torch.float64)
    out[..., :64] = to_fmt(M, fmt).reshape(*M.shape[:-2], 2, 32, 64)
    out[..., 64] = to_fmt(ksum, fmt).reshape(*ksum.shape[:-1], 2, 32)
    return out


def image_to_weight(img, n, k, dtype):
    """inverse of fused_pairs._w_image: 16-bit K-major operand image [K/8][N][8] (bytes) -> (N, K) float64"""
    return img.contiguous().view(dtype).reshape(k // 8, n, 8).permute(1, 0, 2).reshape(n, k).double()


class Weights:
    """the three weight blobs of FusedXcorr._weights(), decoded"""

    def __init__(self, w1a2, w1b2, w2y, fmt):
        dt = DTYPE[fmt]
        w1a2, w1b2, w2y = (w.detach().cpu() for w in (w1a2, w1b2, w2y))
        o = _W0EXT_BYTES
        self.W0ext1 = image_to_weight(w1a2[:o], 128, 144, dt)          # [W0b diag(g1) | W0a | W0b.beta1 - W0a.beta2 | 0]
        self.W2_1 = image_to_weight(w1a2[o:o + _W2_BYTES], 64, 128, dt)  # centred mlp[2]
        self.g2_1 = w1a2[o + _W2_BYTES:o + _W2_BYTES + 256].view(torch.float32).double()
        wkv = image_to_weight(w1b2[:2 * _W64_BYTES], 128, 64, dt)
        self.Wk2, self.Wv2 = wkv[:64], wkv[64:]
        self.Wm2 = image_to_weight(w1b2[2 * _W64_BYTES:], 64, 64, dt)  # centred stage-2 merge
        self.Wq2 = image_to_weight(w2y[:_W64_BYTES], 64, 64, dt)       # q_proj / c
        o = _W64_BYTES
        self.W0ext2 = image_to_weight(w2y[o:o + _W0EXT_BYTES], 128, 144, dt)   # [W0a | W0b diag(g1) | W0b.beta1 | 0]
        o += _W0EXT_BYTES
        self.W2_2 = image_to_weight(w2y[o:o + _W2_BYTES], 64, 128, dt)
        self.g2_2 = w2y[o + _W2_BYTES:o + _W2_BYTES + 256].view(torch.float32).double()

    @classmethod
    def of(cls, fx):
        fx._weights()
        return cls(fx._w1a2, fx._w1b2, fx._w2y, fx.fmt)


def attention_norm(Qf, MK, att_eps, fmt):
    """per-head linear attention of the queries Qf (..., n, 64) against an attention operand MK (..., 2, 32, 80), merged
    (the merge weight is inside MK), LayerNorm without affine -> X' rounded to fmt.  The per-head read-out is
    (Qf_h . M_h) / (Qf_h . Ksum_h + att_eps)."""
    x = 0.0
    for h in range(2):
        q = Qf[..., 32 * h:32 * h + 32]
        acc = q @ MK[..., h, :, :]                                     # (..., n, 80): 64 merged channels | Q.Ksum | 0
        x = x + acc[..., :64] / (acc[..., 64:65] + att_eps)
    return to_fmt(x / torch.sqrt((x * x).mean(-1, keepdim=True) + LN_EPS), fmt)


def ffn(G, W0ext, W2, g2, residual, fmt):
    """G = the K = 129 operand [.. | .. | 1]: hidden = fmt(relu(G W0ext^T)), y = hidden W2^T, residual + g2 * y / rms(y)"""
    hid = to_fmt(torch.relu(G @ W0ext[:, :129].T), fmt)
    y = hid @ W2.T
    return residual + g2 * y / torch.sqrt((y * y).mean(-1, keepdim=True) + LN_EPS)


def _ones(x):
    return torch.ones(*x.shape[:-1], 1, dtype=torch.float64)


def phase1a(QF1, H, MK1, W, att_eps, npts, fmt):
    """pair_p1a2: stage-1 output A (..., npts, 64) of the search object (QF1, H images) against the template operand MK1"""
    QF1, H = QF1[..., :npts, :], H[..., :npts, :]
    X = attention_norm(QF1, MK1, att_eps, fmt)
    return to_fmt(ffn(torch.cat([X, H, _ones(H)], -1), W.W0ext1, W.W2_1, W.g2_1, H, fmt), fmt)


def elu1_keys(k, fmt):
    """the key feature elu(k) + 1 as the phase-1b kernels form it (module docstring)"""
    if fmt == FMT_F16:
        return to_fmt(elu1(k), fmt)
    x = to_fmt(k, fmt)
    e = to_fmt(torch.exp2(to_fmt(torch.clamp(x, max=0.0) * LOG2E_B, fmt)), fmt)
    return to_fmt(torch.clamp(x, min=0.0) + e, fmt)


def phase1b(A, PV, W, kv_scale, npts, fmt):
    """pair_p1b_n: stage-2 attention operand B7 (..., 2, 32, 80) of A (..., >= npts, 64) as template; PV the Wv2 pos image of the
    object A belongs to.  Only rows < npts enter the key / value sums."""
    A, PV = A[..., :npts, :], PV[..., :npts, :]
    Kf = elu1_keys(A @ W.Wk2.T, fmt)
    v = A @ W.Wv2.T
    V = to_fmt((v if fmt == FMT_F16 else to_fmt(v, fmt)) + PV, fmt)
    KV = Kf.transpose(-1, -2) @ V * kv_scale                            # (..., 64 d, 64 v)
    ksum = Kf.sum(-2) * kv_scale
    head = torch.arange(64) // 32
    KVbd = to_fmt(KV * (head[:, None] == head[None, :]), fmt)
    return pack_b7(KVbd @ W.Wm2.T, ksum, fmt)


def query_feature(q, fmt):
    """elu(x) + 1 of the stage-2 queries from the pre-scaled projection q = (Wq / c) a (module docstring)"""
    if fmt == FMT_F16:
        return to_fmt(torch.clamp(q, min=0.0) * math.log(2.0) + torch.exp2(torch.clamp(q, max=0.0)), fmt)
    x = to_fmt(q, fmt)
    return to_fmt(torch.clamp(x, min=0.0) * LN2B + to_fmt(torch.exp2(torch.clamp(x, max=0.0)), fmt), fmt)


def phase2_rows(A, B7, W, att_eps, npts, fmt):
    """stage-2 output o - beta2 (..., npts, 64) of the search rows A against the template operand B7 (fp32 in the kernel)"""
    A = A[..., :npts, :]
    X = attention_norm(query_feature(A @ W.Wq2.T, fmt), B7, att_eps, fmt)
    return ffn(torch.cat([A, X, _ones(A)], -1), W.W0ext2, W.W2_2, W.g2_2, A, fmt)


def phase2(A, B7, W, att_eps, npts, fmt):
    """pair_p2y: pooled partials (..., 128) = [max | sum] over the npts real rows of o - beta2"""
    o = phase2_rows(A, B7, W, att_eps, npts, fmt)
    return torch.cat([o.amax(-2), o.sum(-2)], -1)


def pool_finish(part, npts, beta2):
    """pcreid_pool_finish2: part (P, 2, 128) -> pooled (P, 128): max over both directions | mean over the 2 npts points, + beta2"""
    part = part.double()
    b = beta2.double()
    return torch.cat([torch.maximum(part[:, 0, :64], part[:, 1, :64]) + b,
                      (part[:, 0, 64:] + part[:, 1, 64:]) / (2 * npts) + b], -1)


# --------------------------------------------------------------------------------------------------------------------------
# chaining: per-object fp32 inputs (h, xyz) -> logits, the way FusedXcorr.prepare + match do
# --------------------------------------------------------------------------------------------------------------------------
def _w(p):
    return p.detach().double().cpu()


def _pos_code(X, xyz):
    """pos_mlp(xyz) (B, N, 64); None for token sets without coordinates"""
    if xyz is None:
        return None
    hid = torch.relu(xyz.double() @ _w(X.pos_mlp[0].weight).T + _w(X.pos_mlp[0].bias))
    return hid @ _w(X.pos_mlp[2].weight).T + _w(X.pos_mlp[2].bias)


def kv_scale(fmt, npts):
    """the scale the fp16 format stores key / value sums with (FusedXcorr.kv_scale)"""
    return 1.0 / npts if fmt == FMT_F16 else 1.0


def prepare(model, fmt, h, xyz):
    """FusedXcorr.prepare: h (B, 64, N), xyz (B, N, 3) or None -> dict of decoded per-object operands QF1, H, PV (B, N, 64) and
    MK1 (B, 2, 32, 80).  MK1 = [blockdiag(KV1) Wm1c^T | Ksum1] of the object as stage-1 template, with the merge weight centred over
    its output channels and both parts scaled by kv_scale."""
    X1, X2 = model.cross_stage1, model.cross_stage2
    hp = h.detach().double().cpu().transpose(1, 2)
    N = hp.shape[1]
    QF1 = pack(hp @ _w(X1.q_proj.weight).T, fmt, ACT_ELU1)
    H = pack(hp, fmt, bias=X1.norm2.bias.detach().cpu())
    pos2 = _pos_code(X2, xyz)
    PV = torch.zeros_like(hp) if pos2 is None else to_fmt(pos2 @ _w(X2.v_proj.weight).T, fmt)
    pos1 = _pos_code(X1, xyz)
    Kf = elu1(hp @ _w(X1.k_proj.weight).T)
    V = (hp if pos1 is None else hp + pos1) @ _w(X1.v_proj.weight).T
    head = torch.arange(64) // 32
    KV = (Kf.transpose(1, 2) @ V) * (head[:, None] == head[None, :])
    wm = _w(X1.merge.weight)
    sc = kv_scale(fmt, N)
    MK1 = pack_b7(KV @ (wm - wm.mean(0, keepdim=True)).T * sc, Kf.sum(1) * sc, fmt)
    return dict(QF1=QF1, H=H, PV=PV, MK1=MK1, npts=N)


def match(model, fmt, W, ps, pt, ti, dj):
    """FusedXcorr.match on decoded operands: pairs (ti[p], dj[p]) of the prepared sets ps, pt -> dict A (P, 2, N, 64),
    B7 (P, 2, 2, 32, 80), part (P, 2, 128), pooled (P, 128) (float64)"""
    N = ps["npts"]
    sc = kv_scale(fmt, N)
    ti, dj = torch.as_tensor(ti).long().cpu(), torch.as_tensor(dj).long().cpu()
    sides = ((ps, ti, pt, dj), (pt, dj, ps, ti))                       # role r: (search set, index, template set, index)
    A = torch.stack([phase1a(s["QF1"][i], s["H"][i], t["MK1"][j], W, ATT_EPS * sc, N, fmt) for s, i, t, j in sides], 1)
    B7 = torch.stack([phase1b(A[:, r], s["PV"][i], W, sc, N, fmt) for r, (s, i, _, _) in enumerate(sides)], 1)
    part = torch.stack([phase2(A[:, r], B7[:, 1 - r], W, ATT_EPS * sc, N, fmt) for r in (0, 1)], 1)
    pooled = pool_finish(part, N, model.cross_stage2.norm2.bias.detach().cpu())
    return dict(A=A, B7=B7, part=part, pooled=pooled)
