"""CPU: the float64 reference of the fused matcher (tests/fused_reference.py) chained from per-object inputs, on the weight
blobs FusedXcorr._weights() folds, against the float64 oracle (ReIDNet.xcorr_eff restated over the state_dict): the stage-1
outputs a / b, the max / sum pooling of the stage-2 outputs o1n / o2n, and the logits.  This pins the reference the GPU tests
measure the kernels against, and the host-side weight folding (LayerNorm1 affine, beta2 bias column, centred merge / mlp[2],
pre-scaled q_proj) without a GPU.

Tolerances.  u = unit roundoff of the operand format (fp16 2^-11, bf16 2^-8).  The reference rounds to the format at every
operand the kernels store (about six roundings in a row, each <= u/2 relative, passed through LayerNorms that renormalise them),
so its distance from the exact oracle is a small multiple of u times the tensor's scale:
  tensor (a, b, pooled max, pooled sum):  max|ref - oracle| <= 3 u max|oracle|   measured <= 1.6 u (fp16 1.3 u, bf16 1.6 u)
  logits:                                 max|ref - oracle| <= 4 u               measured <= 1.9 u (fp16 1.4 u, bf16 1.9 u)
A folding error is tens to hundreds of u (test_folding_errors_are_detected: >= 4 u on the weakest comparison in bf16, >= 33 u in
fp16)."""
import functools

import pytest
import torch

import fused_reference as R
import helpers
from oracle import reid_oracle as O

TOL_TENSOR = 3.0        # x u x max|oracle|
TOL_LOGIT = 4.0         # x u
FMTS = {"parity_tc": R.FMT_F16, "fast": R.FMT_BF16}


@functools.lru_cache(maxsize=None)
def _model():
    return helpers.build_pair("pt", (256, 128, 64))


def oracle_chain(orc, h1, x1, h2, x2):
    """float64 oracle (a float64 copy of orc.sd) of one batch of pairs -> stage-1 a, b (B, 64, N), stage-2 o1n, o2n, logits.
    x1 = x2 = None: token sets (cross_lin_attn: the same block without the position code)."""
    sd = {k: v.double() for k, v in orc.sd.items()}
    h1, h2 = h1.double(), h2.double()
    if x1 is None:
        ca = lambda p, s, xs, t, xt: O.cross_lin_attention(sd, p, s, t)
    else:
        x1, x2 = x1.double(), x2.double()
        ca = lambda p, s, xs, t, xt: O.cross_attention(sd, p, s, xs, t, xt)
    a, b = ca("cross_stage1", h1, x1, h2, x2), ca("cross_stage1", h2, x2, h1, x1)
    o1, o2 = ca("cross_stage2", a, x1, b, x2), ca("cross_stage2", b, x2, a, x1)
    return a, b, o1, o2, oracle_head(orc, O.pooled_feats(torch.cat([o1, o2], 2), "both"))


def oracle_head(orc, pooled):
    sd = {k: v.double() for k, v in orc.sd.items() if k.startswith("match_head.")}
    return O._lin(sd, "match_head.1", O.linear_res(sd, "match_head.0", pooled.double(), orc.head_ng)).squeeze(1)


def chain_errors(W, fmt, N, xyz, seed=0):
    """-> {name: error in units of u (tensors: relative to the oracle tensor's max|.|)} of the chained reference on 3 objects,
    all-pairs subset with self-pairs"""
    m, orc = _model()
    g = torch.Generator().manual_seed(seed + N)
    h = torch.randn(3, 64, N, generator=g) * 0.5
    x = O.synth_objects(3, N, seed + N) if xyz else None
    ti, dj = torch.tensor([0, 0, 1, 2, 2, 1]), torch.tensor([0, 1, 2, 1, 0, 1])
    pk = R.prepare(m, fmt, h, x)
    r = R.match(m, fmt, W, pk, pk, ti, dj)
    a, b, o1, o2, lo = oracle_chain(orc, h[ti], None if x is None else x[ti], h[dj], None if x is None else x[dj])
    u = R.UNIT_ROUNDOFF[fmt]
    rel = lambda got, ref: float((got - ref).abs().max() / (u * ref.abs().max()))
    b2 = m.cross_stage2.norm2.bias.detach().double()
    part = r["part"]
    return {"a": rel(r["A"][:, 0], a.transpose(1, 2)), "b": rel(r["A"][:, 1], b.transpose(1, 2)),
            "o1n max": rel(part[:, 0, :64] + b2, o1.amax(2)), "o1n sum": rel(part[:, 0, 64:] + N * b2, o1.sum(2)),
            "o2n max": rel(part[:, 1, :64] + b2, o2.amax(2)), "o2n sum": rel(part[:, 1, 64:] + N * b2, o2.sum(2)),
            "logit": float((oracle_head(orc, r["pooled"]) - lo).abs().max()) / u}


def _fails(errs):
    return {k: v for k, v in errs.items() if v > (TOL_LOGIT if k == "logit" else TOL_TENSOR)}


@pytest.mark.parametrize("xyz", [True, False], ids=["points", "tokens"])
@pytest.mark.parametrize("N", [1, 2, 129, 256])
@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
def test_reference_chain_matches_oracle(mode, N, xyz):
    from pcreid_b200.models import fused_pairs
    fmt = FMTS[mode]
    W = R.Weights.of(fused_pairs.FusedXcorr(_model()[0], fmt))
    errs = chain_errors(W, fmt, N, xyz)
    assert not _fails(errs), f"{mode} N={N}: reference off the oracle (units of u): {errs}"


def _broken_weights(fx, fold):
    """the blobs of fx with one folded term broken: 'bias1' drops -W0a.beta2 from stage 1's bias column, 'gamma1' drops the
    LayerNorm1 gamma column scaling of stage 1, 'center1' / 'center2' leave mlp[2] of stage 1 / 2 uncentred"""
    from pcreid_b200.models import fused_pairs as FP
    fx._weights()
    X1, X2 = fx.model.cross_stage1, fx.model.cross_stage2
    f = lambda t: t.detach().float()
    w1a2, w2y = fx._w1a2.clone(), fx._w2y.clone()
    W0 = f(X1.mlp[0].weight)
    W0ext = torch.zeros(128, 144)
    W0ext[:, :64] = W0[:, 64:] * (1.0 if fold == "gamma1" else f(X1.norm1.weight)[None, :])
    W0ext[:, 64:128] = W0[:, :64]
    W0ext[:, 128] = W0[:, 64:] @ f(X1.norm1.bias) - (0.0 if fold == "bias1" else W0[:, :64] @ f(X1.norm2.bias))
    w1a2[:W0ext.numel() * 2] = FP._w_image(W0ext, fx.dtype)
    w2 = 128 * 144 * 2
    if fold == "center1":
        w1a2[w2:w2 + 16384] = FP._w_image(f(X1.mlp[2].weight), fx.dtype)
    if fold == "center2":
        w2 += 8192
        w2y[w2:w2 + 16384] = FP._w_image(f(X2.mlp[2].weight), fx.dtype)
    return R.Weights(w1a2, fx._w1b2, w2y, fx.fmt)


@pytest.mark.parametrize("fold", ["none", "bias1", "gamma1", "center1", "center2"])
@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
def test_folding_errors_are_detected(mode, fold):
    """one broken folded term in the weight blobs must fail the oracle comparison of test_reference_chain_matches_oracle (the
    tolerances tell a folding bug from rounding); 'none' rebuilds the blobs unbroken and must pass, and equal _weights() bit for bit"""
    from pcreid_b200.models import fused_pairs
    fx = fused_pairs.FusedXcorr(_model()[0], FMTS[mode])
    W = _broken_weights(fx, fold)
    if fold == "none":
        ref = R.Weights.of(fx)
        assert all(torch.equal(getattr(W, k), getattr(ref, k)) for k in vars(ref))
    for N in (2, 129):
        fails = _fails(chain_errors(W, fx.fmt, N, True))
        assert bool(fails) == (fold != "none"), f"{mode} {fold} N={N}: failing comparisons {fails}"


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
def test_weight_blob_decoding(mode):
    """the decoded blobs are the folded weights of the model, rounded to the format"""
    from pcreid_b200.models import fused_pairs
    m, _ = _model()
    fmt = FMTS[mode]
    fx = fused_pairs.FusedXcorr(m, fmt)
    W = R.Weights.of(fx)
    X1, X2 = m.cross_stage1, m.cross_stage2
    d = lambda t: t.detach().double()
    c = lambda w: d(w) - d(w).mean(0, keepdim=True)
    close = lambda got, ref: float((got - ref).abs().max()) <= R.UNIT_ROUNDOFF[fmt] * float(ref.abs().max())
    assert close(W.W0ext1[:, :64], d(X1.mlp[0].weight)[:, 64:] * d(X1.norm1.weight))
    assert close(W.W0ext1[:, 64:128], d(X1.mlp[0].weight)[:, :64])
    assert close(W.W2_1, c(X1.mlp[2].weight)) and close(W.W2_2, c(X2.mlp[2].weight)) and close(W.Wm2, c(X2.merge.weight))
    assert close(W.Wk2, d(X2.k_proj.weight)) and close(W.Wv2, d(X2.v_proj.weight))
    assert close(W.W0ext2[:, :64], d(X2.mlp[0].weight)[:, :64])
    assert close(W.W0ext2[:, 128], d(X2.mlp[0].weight)[:, 64:] @ d(X2.norm1.bias))
    ln2 = R.LN2B if fmt == R.FMT_BF16 else 0.6931471805599453
    assert close(W.Wq2, d(X2.q_proj.weight) / ln2)
    assert torch.equal(W.g2_1, d(X1.norm2.weight)) and torch.equal(W.g2_2, d(X2.norm2.weight))
    assert (W.W0ext1[:, 129:] == 0).all() and (W.W0ext2[:, 129:] == 0).all()
