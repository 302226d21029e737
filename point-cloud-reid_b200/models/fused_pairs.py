"""Host side of the fused tensor-core `xcorr_eff` matcher (csrc/pair_tc.cu, csrc/pair_tc2.cu) -- the tensor-core
modes of ReIDNet.match_all_pairs / match_forward_inference:

  'fast'      bf16 operand images (8-bit significand), |dlogit| <= 3e-2
  'parity_tc' fp16 operand images (11-bit significand, the precision of tf32 at the tensor-pipe rate and operand bytes of
              bf16), |dlogit| <= 5e-3.  fp16's narrow exponent is safe here because every operand is O(1) by construction:
              LayerNorm outputs, elu+1 features, projections of those, and key/value sums that are stored divided by the
              point count (the attention read-out is a ratio, so the scale cancels; LinearAttention's eps is scaled
              with it).  Conversions saturate instead of overflowing.
              Feature range: tests/test_gpu_fused_phases.py sweeps the search / template features h from 1/16 to 16 times
              the encoder's scale (max|h| ~ 2): both modes stay inside their gates (parity_tc |dlogit| 3.1e-3, fast 1.1e-2 at
              x16 on an NVIDIA B200).  The largest fp16 operand grows as the square of that scale (the unnormalised
              key/value products of the stage-1 attention operand, max ~ 0.75 at x1), so fp16 saturation is estimated to begin
              near x300 (not exercised by the tests).

Everything that depends on one object only is computed once per object with the fp32 kernels and packed to 16-bit
operand images (stage-1 queries elu(Wq1 h)+1, h + beta2, Wv2 pos2(xyz), and the stage-1 attention operand
MK1 = [head-split blockdiag(KV1) Wm1^T | Ksum1]); the three fused kernels then score pairs without writing any per-pair
activation except the 16-bit stage-1 outputs (64 KB / pair at 256 points) and the stage-2 attention operands (20 KB / pair).
Reference: ReIDNet.xcorr_eff + get_pooled_feats + match_head (mmdet3d/models/ReIDNet.py:231-247, 526-534, 444-453).
"""
import math
import os

import torch

from .. import kernels as K
from .. import torch_ops as _T
from ._packing import kmajor

IMG = 16384
# attention operand: one [10 n-chunks][32 k][8] 16-bit image per head (pair_common.cuh B7_BYTES; the override exists for A/B runs
# against an older build of the library, scripts/gpu_prev_ab.sh)
B7_BYTES = int(os.environ.get("PCREID_B7_BYTES", 10240))
FMT_BF16, FMT_F16 = 0, 1
LN2H = 0.693359375        # f16(ln 2): the same for the packed f16x2 A/B build (PCREID_F16_PACKED=1)
LN2B = 0.69140625          # bf16(ln 2): the packed elu epilogue of the bf16 kernels multiplies by this constant
ATT_EPS = 1e-6             # LinearAttention.eps (attention.py:21)


def _center_out(w):
    """(out, in) weight minus its mean over the output axis: the Linear's output has zero mean over channels, so the
    LayerNorm that follows needs no mean (LayerNorm is invariant to a per-row shift of its input)."""
    w = w.detach().float()
    return w - w.mean(0, keepdim=True)


_OPS = _T.ops          # torch.ops.pcreid.*


def _w_image(w, dtype):
    """torch weight (N, K) -> 16-bit K-major operand image [K/8][N][8] as bytes."""
    N, Kd = w.shape
    return w.detach().to(dtype).view(N, Kd // 8, 8).permute(1, 0, 2).contiguous().view(torch.uint8).flatten()


def _f32_bytes(*ts):
    return torch.cat([t.detach().float().flatten() for t in ts]).contiguous().view(torch.uint8)


def supported(model, n_points):
    X1, X2 = model.cross_stage1, model.cross_stage2
    return (model.match_type == 'xcorr_eff' and model.combine == 'point-cat' and model.pool_type == 'both'
            and X1 is not None and X2 is not None and X1.q_proj.weight.shape == (64, 64) and X1.nhead == 2
            and X2.q_proj.weight.shape == (64, 64) and X2.nhead == 2 and n_points >= 1)


class ObjectPack:
    """per-object operand images of a set of objects (tracks or detections)."""
    __slots__ = ("n", "npts", "fmt", "QF1", "H", "PV", "MK1")


class FusedXcorr:
    def __init__(self, model, fmt=FMT_BF16):
        self.model = model
        self.fmt = fmt
        self.dtype = torch.float16 if fmt == FMT_F16 else torch.bfloat16
        self._key = None
        self.n_ctas = None
        self._n_ctas_dev = None
        self.timing = None      # set to a list to collect (name, start_event, end_event) per fused kernel launch
        self._units = {}        # dense-block unit lists by geometry (see _dense_units)

    def _weights(self):
        X1, X2 = self.model.cross_stage1, self.model.cross_stage2
        key = tuple((t.data_ptr(), t._version) for t in list(X1.parameters()) + list(X2.parameters()))
        if key != self._key:
            with torch.no_grad():
                d, dt = 64, self.dtype
                # LN1 affine folded forward, centred merge / mlp[2], q_proj scaled for the exp2-based elu epilogue
                f = lambda t: t.detach().float()
                W0_1, W0_2 = f(X1.mlp[0].weight), f(X2.mlp[0].weight)
                # stage 1, G2 operand [X' | h + beta2 | 1]: columns = W0b.diag(g1) | W0a | W0b.beta1 - W0a.beta2 (the residual image
                # carries LayerNorm2's beta, so the constant it adds through W0a is taken back out in the bias column)
                self._b2_1 = f(X1.norm2.bias).contiguous()                         # added to the residual image H
                W0ext1 = torch.zeros((2 * d, 2 * d + 16), device=W0_1.device)
                W0ext1[:, :d] = W0_1[:, d:] * f(X1.norm1.weight)[None, :]
                W0ext1[:, d:2 * d] = W0_1[:, :d]
                W0ext1[:, 2 * d] = W0_1[:, d:] @ f(X1.norm1.bias) - W0_1[:, :d] @ self._b2_1
                self._w1a2 = torch.cat([
                    _w_image(W0ext1, dt), _w_image(_center_out(X1.mlp[2].weight), dt), _f32_bytes(X1.norm2.weight)]).contiguous()
                self._merge1c = kmajor(_center_out(X1.merge.weight))
                self._w1b2 = torch.cat([
                    _w_image(torch.cat([X2.k_proj.weight, X2.v_proj.weight], 0), dt),
                    _w_image(_center_out(X2.merge.weight), dt)]).contiguous()
                W0ext = torch.zeros((2 * d, 2 * d + 16), device=W0_2.device)
                W0ext[:, :d] = W0_2[:, :d]
                W0ext[:, d:2 * d] = W0_2[:, d:] * f(X2.norm1.weight)[None, :]
                W0ext[:, 2 * d] = W0_2[:, d:] @ f(X2.norm1.bias)
                ln2 = (LN2H if os.environ.get("PCREID_F16_PACKED") == "1" else math.log(2.0)) if self.fmt == FMT_F16 else LN2B
                self._w2y = torch.cat([
                    _w_image(f(X2.q_proj.weight) / ln2, dt), _w_image(W0ext, dt), _w_image(_center_out(X2.mlp[2].weight), dt),
                    _f32_bytes(X2.norm2.weight)]).contiguous()
                self._b2_2 = f(X2.norm2.bias).contiguous()                         # added after the pooling
                assert self._w1a2.numel() == 53504 and self._w2y.numel() == 61696 and self._w1b2.numel() == 24576
            self._key = key

    def _tick(self):
        if self.timing is None:
            return None
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def _tock(self, name, e0, units):
        if e0 is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            self.timing.append((name, e0, e1, units))

    def _pack_image(self, x, act=K.ACT_NONE):
        B, C, N = x.shape
        out = torch.empty((B, (N + 127) // 128, C // 8, 128, 16), device=x.device, dtype=torch.uint8)
        _OPS.pack_image(B, C, N, x, x.stride(0), x.stride(1), act, self.fmt, out)
        return out

    def kv_scale(self, npts):
        """scale the key/value sums of a template with `npts` points are stored with (fp16: 1/points keeps them O(1))."""
        return 1.0 / npts if self.fmt == FMT_F16 else 1.0

    def prepare(self, h, xyz):
        """h (B, 64, N) fp32 channel-major, xyz (B, N, 3) (None for token sets without coordinates) -> ObjectPack."""
        X1, X2 = self.model.cross_stage1, self.model.cross_stage2
        pk1, pk2 = X1.packed(), X2.packed()
        self._weights()
        B, C, N = h.shape
        o = ObjectPack()
        o.n, o.npts, o.fmt = B, N, self.fmt
        o.QF1 = self._pack_image(K.cn_linear(h, pk1["q"]), K.ACT_ELU1)
        o.H = torch.empty((B, (N + 127) // 128, C // 8, 128, 16), device=h.device, dtype=torch.uint8)
        _OPS.pack_image_bias(B, C, N, h, h.stride(0), h.stride(1), self._b2_1, self.fmt, o.H)   # h + beta2
        pos2 = X2.position_code(xyz)
        if pos2 is None:            # cross_lin_attn (image tokens, attention.py:312-372): no position code -> Wv.pos == 0
            o.PV = torch.zeros((B, (N + 127) // 128, C // 8, 128, 16), device=h.device, dtype=torch.uint8)
        else:
            o.PV = self._pack_image(K.cn_linear(pos2, pk2["v"]))
        wkv, ksum = X1.template_summary(h, X1.position_code(xyz))          # (B, 64, 64) [d][v] block diagonal, (B, 64)
        M = K.cn_linear(wkv, self._merge1c, x1_pm=True, y_pm=True)          # (B, d, out) = blockdiag(KV) Wm^T
        # template_summary follows the reference's values / S (attention.py:47): M carries 1/N, ksum does not
        sc = self.kv_scale(N)
        M.mul_(float(N) * sc)
        if sc != 1.0:
            ksum = ksum * sc
        o.MK1 = torch.empty((B, B7_BYTES), device=h.device, dtype=torch.uint8)
        _OPS.pack_b7(B, M, ksum, self.fmt, o.MK1)
        return o

    def _dense_units(self, dev, r0, nrows, Dn, by_search, b_by_search):
        """(search, template, slot) int32 lists of the row block [r0, r0 + nrows) x [0, Dn), per role, in the orders phase 1a and
        phase 1b want.  They depend on the block's geometry only, so a steady stream of equal-shaped matches (the chunks of a large
        matrix, a tracker's frames) reuses them instead of re-running ~25 index kernels per chunk; never cached while a CUDA graph
        is being captured (the tensors would live in the graph's private pool)."""
        key = (str(dev), r0, nrows, Dn, by_search, b_by_search)
        capturing = torch.cuda.is_current_stream_capturing()      # a graph must own every buffer its kernels read: no cache either way
        hit = None if capturing else self._units.get(key)
        if hit is not None:
            return hit
        P = nrows * Dn
        u = torch.arange(P, device=dev, dtype=torch.int32)
        t_of, d_of = r0 + u % nrows, u // nrows
        c = lambda *xs: tuple(x.contiguous() for x in xs)
        lists_s = (c(r0 + u // Dn, u % Dn, u),                                        # role 0 (search, template, slot): row-major
                   c(u // nrows, r0 + u % nrows, (u % nrows) * Dn + u // nrows))       # role 1: detection-major
        lists_t = (c(t_of, d_of, (t_of - r0) * Dn + d_of),                             # role 0: runs of equal detection (template)
                   c(u % Dn, r0 + u // Dn, u))                                        # role 1: row-major = sorted by track (template)
        out = (lists_s if by_search else lists_t, lists_s if b_by_search else lists_t)
        if not capturing:
            if len(self._units) >= 64:                      # a few MB per entry: keep the working set of one large matrix
                self._units.pop(next(iter(self._units)))
            self._units[key] = out
        return out

    def match(self, pt, pd, ti, dj, debug=None, dense=None):
        """logits (P,) for the pairs (ti[p], dj[p]); ti / dj int64 or int32 index tensors on the device.
        dense=(r0, nrows, D): the pairs are the full row block [r0, r0+nrows) x [0, D) in row-major order (ti, dj may be
        None) -- the unit lists are then generated arithmetically instead of by a stable argsort over the templates."""
        assert pt.npts == pd.npts, "fused matcher expects equal point counts on both sides"
        assert pt.fmt == self.fmt and pd.fmt == self.fmt, "object packs were prepared for another operand format"
        self._weights()
        dev = pt.H.device
        if self.n_ctas is None or self._n_ctas_dev != dev:          # SM count of the device the operands live on
            self.n_ctas, self._n_ctas_dev = torch.cuda.get_device_properties(dev).multi_processor_count, dev
        # unit order: phase 1a keeps the TEMPLATE operand in shared memory across units -> runs of equal template; phase 1b reads
        # per-pair images by slot and the search object's position term -> runs of equal search object, slots ascending
        # (-3.5 ... -5 % on pair_p1b, profiles/r02_unit_order_ab.json; A/B: PCREID_P1B_ORDER=templ)
        by_search = False
        b_by_search = os.environ.get("PCREID_P1B_ORDER", "search") == "search"
        if dense is not None:
            r0, nrows, Dn = dense
            P = nrows * Dn
            unit_lists, unit_lists_b = self._dense_units(dev, r0, nrows, Dn, by_search, b_by_search)
        else:
            P = ti.numel()
            ti, dj = ti.long(), dj.long()
            unit_lists = None
        NT, N = (pt.npts + 127) // 128, pt.npts
        A = torch.empty((P, 2, NT, IMG), device=dev, dtype=torch.uint8)
        B7 = torch.empty((P, 2, B7_BYTES), device=dev, dtype=torch.uint8)
        part = torch.empty((P, 2, 128), device=dev, dtype=torch.float32)
        sc = self.kv_scale(N)
        for role, (srch, tmpl, ps, pm) in enumerate(((ti, dj, pt, pd), (dj, ti, pd, pt))):
            if unit_lists is not None:
                us, ut, sl = unit_lists[role]
                bs, bt, bl = unit_lists_b[role]
            else:
                order = torch.argsort(tmpl, stable=True)                    # phase 1a: runs of units share the template operand
                us, ut, sl = srch[order].int().contiguous(), tmpl[order].int().contiguous(), order.int().contiguous()
                bs, bt, bl = us, ut, sl
                if b_by_search:                                             # phase 1b: runs of units share the search object
                    order = torch.argsort(srch, stable=True)
                    bs, bt, bl = srch[order].int().contiguous(), tmpl[order].int().contiguous(), order.int().contiguous()
            e0 = self._tick()
            _OPS.pair_p1a2(P, N, role, self.fmt, ATT_EPS * sc, us, ut, sl, ps.QF1, ps.H, pm.MK1, self._w1a2, A, self.n_ctas)
            self._tock("pair_p1a2_kernel", e0, P)
            e0 = self._tick()
            _OPS.pair_p1b_n(P, N, role, self.fmt, sc, bs, bt, bl, ps.PV, self._w1b2, A, B7, self.n_ctas)
            self._tock("pair_p1b_kernel" if os.environ.get("PCREID_P1B") == "1" else "pair_p1b2_kernel", e0, P)
        slots = torch.arange(P, device=dev, dtype=torch.int32)
        pooled = torch.empty((1, 128, P), device=dev, dtype=torch.float32)
        for role in (0, 1):
            e0 = self._tick()
            _OPS.pair_p2y(P, N, role, self.fmt, ATT_EPS * sc, slots, A, B7, self._w2y, part, self.n_ctas)
            self._tock("pair_p2y_kernel", e0, P)
        _OPS.pool_finish2(P, N, part, self._b2_2, pooled)
        if debug is not None:
            debug.update(A=A, B7=B7, part=part, pooled=pooled)
        return self.model._head_cn(pooled)


def decode_image(img, dtype=torch.bfloat16):
    """(..., C/8, 128, 16) uint8 operand image -> (..., C, 128) fp32 (debug / tests)."""
    x = img.contiguous().view(dtype).float().transpose(-1, -2)     # (..., C/8, 8, 128)
    return x.reshape(*x.shape[:-3], x.shape[-3] * 8, 128)


def decode_b7(img, dtype=torch.bfloat16):
    """(..., 10240) uint8 attention operand -> (..., 2 heads, 32 k, 80 n) fp32 (debug / tests): n < 64 merged output channels,
    n = 64 the head's Ksum entry."""
    x = img.contiguous().view(dtype).float().reshape(*img.shape[:-1], 2, 10, 32, 8)   # [head][n/8][k][8]
    nd = x.dim()
    return x.permute(*range(nd - 3), nd - 2, nd - 3, nd - 1).reshape(*img.shape[:-1], 2, 32, 80)
