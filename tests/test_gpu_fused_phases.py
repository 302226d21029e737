"""-m gpu: every kernel of the fused `xcorr_eff` matcher (pack_image, pack_image_bias, pack_b7 -> pair_p1a2 -> pair_p1b_n ->
pair_p2y -> pool_finish2) against the float64 reference of tests/fused_reference.py, each on its OWN decoded inputs: the
per-object images of FusedXcorr.prepare and the stored intermediates A (stage-1 output), B7 (stage-2 attention operand) and part
(pooled partials) that FusedXcorr.match(..., debug=) returns.  The inputs of a phase are exact, so its error is its own, and a
failing check names the phase that broke; the logit-only checks of test_gpu_fused.py cannot see a constant per-group offset
(removed by the head's GroupNorm), an error in a non-maximal point, or one divided by 2 npts in the mean.

Tolerances, u = unit roundoff of the operand format (fp16 2^-11, bf16 2^-8).  A phase output is the float64 result rounded to the
format; the kernel accumulates in fp32 and uses approximate ex2 / rsqrt, which moves a value across a rounding boundary of an
intermediate operand now and then (one ulp of X' or of the hidden layer, carried through a 64- or 128-term product, then rounded
once more).  Measured maxima over every case of this file on an NVIDIA B200 (1000 W power limit), fp16 / bf16:
  A  (phase 1a), elementwise / (u (|ref| + rms of the reference row)):  <= 4   measured 2.4 / 2.0
  B7 (phase 1b), the same measure:                                       <= 6   measured 1.5 / 2.9  (two stored roundings in a row:
                                                                                blockdiag(KV), then B7 itself)
  part (phase 2), / (u max|ref|) per half (max | sum):                    <= 1   measured 0.16 / 0.27 (fp32 output: only the
                                                                                roundings inside the phase)
  pooled (pool_finish2), / max|ref|, fp32 arithmetic:                     <= 2^-21 (4 fp32 ulps)   measured 6.6e-8
Against the float64 oracle (the whole chain; derivation in tests/test_fused_reference.py):
  a, b, pooled max / sum, / (u max|oracle|):  <= 3     measured 1.7 / 2.1 (the reference chain alone: 1.3 / 1.6)
  logits, / u:                                <= 4     measured 1.6 / 2.5 at the encoder's feature scale
  logits, feature magnitude sweep:            the mode's gate (5e-3 / 3e-2): the error grows with the logits' scale,
                                              measured 3.1e-3 / 1.1e-2 at h x 16."""
import functools

import pytest
import torch

import fused_reference as R
import helpers
from oracle import reid_oracle as O
from test_fused_reference import TOL_LOGIT, TOL_TENSOR, oracle_chain

pytestmark = pytest.mark.gpu
DEV = "cuda"
FMTS = {"parity_tc": R.FMT_F16, "fast": R.FMT_BF16}
TOL_PHASE = {"A": 4.0, "B7": 6.0, "part": 1.0}
GATE = {R.FMT_F16: 5e-3, R.FMT_BF16: 3e-2}     # the modes' logit gates (test_gpu_fused.py)
TOL_POOLED = 2.0 ** -21


@functools.lru_cache(maxsize=None)
def _pair(kind="pt"):
    if kind == "image":
        return helpers.build_image_pair(192, 64, device=DEV)
    return helpers.build_pair("pt", (256, 128, 64), device=DEV)


def _fused():
    from pcreid_b200.models import fused_pairs
    return fused_pairs


def _objects(B, N, seed, scale=1.0, kind="random", xyz=True):
    """synthetic per-object inputs: h (B, 64, N) ~ 0.5 N(0, 1) * scale (max|h| ~ 2, the encoder's range), xyz (B, N, 3).
    kind 'same': every point of an object identical; 'zero': all-zero h (an empty crop, pc_utils.py:84-89)"""
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(B, 64, N, generator=g) * (0.5 * scale)
    x = O.synth_objects(B, N, seed)
    if kind == "same":
        h = h[:, :, :1].expand(B, 64, N).contiguous()
        x = x[:, :1].expand(B, N, 3).contiguous()
    elif kind == "zero":
        h.zero_()
    return h, (x if xyz else None)


def _rows(img, fmt, npts=None):
    """operand images (..., NT, 8, 128, 16) or (..., NT, 16384) bytes -> (..., points, 64) float64 on the host"""
    if img.shape[-1] == 16384:
        img = img.reshape(*img.shape[:-1], 8, 128, 16)
    x = _fused().decode_image(img, R.DTYPE[fmt]).transpose(-1, -2).flatten(-3, -2).double().cpu()   # (..., NT 128, 64)
    return x if npts is None else x[..., :npts, :]


def _b7(img, fmt):
    return _fused().decode_b7(img, R.DTYPE[fmt]).double().cpu()


def _run(m, fmt, objs_t, objs_d, ti, dj, n_ctas=None, dense=None):
    """prepare + match with the debug intermediates; objs_d None: the template set is the search set (pt is pd)"""
    FP = _fused()
    fx = FP.FusedXcorr(m, fmt)
    pt = fx.prepare(objs_t[0].to(DEV), None if objs_t[1] is None else objs_t[1].to(DEV))
    pd = pt if objs_d is None else fx.prepare(objs_d[0].to(DEV), None if objs_d[1] is None else objs_d[1].to(DEV))
    if n_ctas is not None:
        fx.n_ctas, fx._n_ctas_dev = n_ctas, pt.H.device
    dbg = {}
    if dense is not None:
        L = fx.match(pt, pd, None, None, debug=dbg, dense=dense)
    else:
        L = fx.match(pt, pd, ti.to(DEV), dj.to(DEV), debug=dbg)
    torch.cuda.synchronize()
    return fx, pt, pd, dbg, L


def _elem_err(got, ref, u):
    """max |got - ref| / (u (|ref| + rms of the reference row))"""
    rms = ref.pow(2).mean(-1, keepdim=True).sqrt()
    return float(((got - ref).abs() / (u * (ref.abs() + rms) + 1e-300)).max())


def check_phases(fx, pt, pd, ti, dj, dbg, what=""):
    """each phase of one match against the reference on the GPU's own decoded inputs; -> {check: measured error}"""
    fmt, N = fx.fmt, pt.npts
    u, sc, W = R.UNIT_ROUNDOFF[fmt], fx.kv_scale(N), R.Weights.of(fx)
    obj = [dict(QF1=_rows(o.QF1, fmt, N), H=_rows(o.H, fmt, N), PV=_rows(o.PV, fmt, N), MK1=_b7(o.MK1, fmt)) for o in (pt, pd)]
    A, B7, part = _rows(dbg["A"], fmt, N), _b7(dbg["B7"], fmt), dbg["part"].double().cpu()
    ti, dj = ti.long().cpu(), dj.long().cpu()
    errs = {}
    for r, (s, i, t, j) in enumerate(((obj[0], ti, obj[1], dj), (obj[1], dj, obj[0], ti))):
        A_ref = R.phase1a(s["QF1"][i], s["H"][i], t["MK1"][j], W, R.ATT_EPS * sc, N, fmt)
        errs[f"A role {r}"] = _elem_err(A[:, r], A_ref, u)
        B7_ref = R.phase1b(A[:, r], s["PV"][i], W, sc, N, fmt)
        errs[f"B7 role {r}"] = _elem_err(B7[:, r].flatten(-3, -2), B7_ref.flatten(-3, -2), u)
        p_ref = R.phase2(A[:, r], B7[:, 1 - r], W, R.ATT_EPS * sc, N, fmt)
        for k, sl in (("max", slice(0, 64)), ("sum", slice(64, 128))):
            errs[f"part {k} role {r}"] = float((part[:, r, sl] - p_ref[:, sl]).abs().max() / (u * p_ref[:, sl].abs().max()))
    pooled = dbg["pooled"][0].t().double().cpu()
    p_ref = R.pool_finish(part, N, fx._b2_2.cpu())
    errs["pooled"] = float((pooled - p_ref).abs().max() / p_ref.abs().max())
    bad = {k: v for k, v in errs.items()
           if v > (TOL_POOLED if k == "pooled" else TOL_PHASE["A" if k[0] == "A" else "B7" if k[0] == "B" else "part"])}
    assert not bad, f"{what}: phases off the reference: {bad}"
    return errs


def check_oracle(fx, orc, objs_t, objs_d, ti, dj, dbg, L, what="", logit_tol=None):
    """the whole chain against the float64 oracle: A vs a / b, part + beta2 vs the max / sum of o1n / o2n, logits (within
    TOL_LOGIT u, or the absolute logit_tol)"""
    fmt, N = fx.fmt, objs_t[0].shape[2]
    u = R.UNIT_ROUNDOFF[fmt]
    objs_d = objs_t if objs_d is None else objs_d
    ti, dj = ti.long().cpu(), dj.long().cpu()
    sel = lambda x, i: None if x is None else x[i]
    a, b, o1, o2, lo = oracle_chain(orc, objs_t[0][ti], sel(objs_t[1], ti), objs_d[0][dj], sel(objs_d[1], dj))
    A, part = _rows(dbg["A"], fmt, N), dbg["part"].double().cpu()
    b2 = fx._b2_2.double().cpu()
    rel = lambda got, ref: float((got - ref).abs().max() / (u * ref.abs().max()))
    errs = {"a": rel(A[:, 0], a.transpose(1, 2)), "b": rel(A[:, 1], b.transpose(1, 2))}
    for r, o in enumerate((o1, o2)):
        errs[f"max role {r}"] = rel(part[:, r, :64] + b2, o.amax(2))
        errs[f"sum role {r}"] = rel(part[:, r, 64:] + N * b2, o.sum(2))
    errs["logit"] = float((L.double().cpu() - lo).abs().max()) / u
    lt = TOL_LOGIT if logit_tol is None else logit_tol / u
    bad = {k: v for k, v in errs.items() if v > (lt if k == "logit" else TOL_TENSOR)}
    assert not bad, f"{what}: chain off the float64 oracle (units of u): {bad}"
    return errs


# ---------------------------------------------------------------------------------------------------------------------------
# a. packers, bit for bit
# ---------------------------------------------------------------------------------------------------------------------------
def _strided(B, C, N, seed, big=None):
    """(B, C, N) fp32 view with a non-dense batch stride and a row stride lds > N"""
    g = torch.Generator().manual_seed(seed)
    base = torch.randn(B, C + 16, N + 37, generator=g) * 2.0
    if big is not None:
        base[:, :, ::5] = big
        base[:, :, 1::5] = -big
    return base.to(DEV)[:, 8:8 + C, 3:3 + N]


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("N", [1, 127, 128, 129, 300])
def test_pack_images_match_reference(N, mode):
    """pack_image (plain and elu+1) and pack_image_bias from strided sources: real rows equal the reference's rounding (elu+1:
    within one ulp -- the kernel's expf and fp32 +1 each round once more), padding rows are zero, every byte is written"""
    FP = _fused()
    fmt, B, C = FMTS[mode], 3, 64
    NT = (N + 127) // 128
    x = _strided(B, C, N, N)
    assert not x.is_contiguous() and x.stride(1) > N and x.stride(0) > C * x.stride(1)
    bias = torch.randn(C, generator=torch.Generator().manual_seed(1)).to(DEV)
    ref_rows = lambda **kw: R.pack(x.double().cpu().transpose(1, 2), fmt, **kw)
    for act in (R.ACT_NONE, R.ACT_ELU1, "bias"):
        out = torch.full((B, NT, C // 8, 128, 16), 0xAB, dtype=torch.uint8, device=DEV)
        if act == "bias":
            FP._OPS.pack_image_bias(B, C, N, x, x.stride(0), x.stride(1), bias, fmt, out)
            ref = R.pack(x.double().cpu().transpose(1, 2), fmt, bias=bias.cpu())
        else:
            FP._OPS.pack_image(B, C, N, x, x.stride(0), x.stride(1), act, fmt, out)
            ref = ref_rows(act=act)
        got = _rows(out, fmt)
        assert (got[:, N:] == 0).all(), f"{act}: padding rows not zero"
        got = got[:, :N]
        if act == R.ACT_ELU1:          # elu + 1 > 0: adjacent 16-bit patterns are one ulp apart
            bits = lambda t: t.to(R.DTYPE[fmt]).view(torch.int16).int()
            assert (bits(got) - bits(ref)).abs().max() <= 1
        else:
            assert torch.equal(got, ref), f"{act}: {int((got != ref).sum())} elements differ"


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
def test_pack_saturation(mode):
    """fp16 conversions saturate: +-1e6 packs to +-65504 (a plain fp16 cast gives inf); bf16 keeps the value's magnitude"""
    FP = _fused()
    fmt, B, C, N = FMTS[mode], 2, 64, 129
    x = _strided(B, C, N, 5, big=1e6)
    bias = torch.zeros(C, device=DEV)
    for fn in ("pack_image", "pack_image_bias"):
        out = torch.zeros((B, 2, C // 8, 128, 16), dtype=torch.uint8, device=DEV)
        if fn == "pack_image":
            FP._OPS.pack_image(B, C, N, x, x.stride(0), x.stride(1), R.ACT_NONE, fmt, out)
        else:
            FP._OPS.pack_image_bias(B, C, N, x, x.stride(0), x.stride(1), bias, fmt, out)
        got = _rows(out, fmt, N)
        ref = R.pack(x.double().cpu().transpose(1, 2), fmt)
        assert torch.isfinite(got).all() and torch.equal(got, ref), fn
        if fmt == R.FMT_F16:
            assert got.abs().max() == 65504.0 and torch.isinf(x.half()).any()
    M = torch.full((B, 64, 64), 1e6, device=DEV)
    M[:, :, ::2] = -1e6
    out = torch.zeros((B, 10240), dtype=torch.uint8, device=DEV)
    FP._OPS.pack_b7(B, M, torch.full((B, 64), 1e6, device=DEV), fmt, out)
    got = _b7(out, fmt)
    assert torch.isfinite(got).all() and torch.equal(got, R.pack_b7(M.double().cpu(), torch.full((B, 64), 1e6).double(), fmt))


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("B", [1, 5])
def test_pack_b7_matches_reference(B, mode):
    """pack_b7: per head the 32 rows of M and Ksum, columns 65..79 zero, every byte written"""
    FP = _fused()
    fmt = FMTS[mode]
    g = torch.Generator().manual_seed(B)
    M, ks = torch.randn(B, 64, 64, generator=g).to(DEV), (torch.rand(B, 64, generator=g) * 50).to(DEV)
    out = torch.full((B, 10240), 0xAB, dtype=torch.uint8, device=DEV)
    FP._OPS.pack_b7(B, M, ks, fmt, out)
    assert torch.equal(_b7(out, fmt), R.pack_b7(M.double().cpu(), ks.double().cpu(), fmt))


@pytest.mark.parametrize("P", [1, 37, 100])
@pytest.mark.parametrize("npts", [1, 129, 256])
def test_pool_finish_matches_reference(npts, P):
    """pool_finish2: max over both directions | (sum0 + sum1) / (2 npts), + beta2 (or no bias)"""
    FP = _fused()
    g = torch.Generator().manual_seed(P + npts)
    part = (torch.randn(P, 2, 128, generator=g) * torch.tensor([1.0] * 64 + [float(npts)] * 64)).to(DEV)
    bias = torch.randn(64, generator=g).to(DEV)
    for b in (bias, None):
        out = torch.full((1, 128, P), float("nan"), device=DEV)
        FP._OPS.pool_finish2(P, npts, part, b, out)
        ref = R.pool_finish(part.cpu(), npts, torch.zeros(64) if b is None else b.cpu())
        got = out[0].t().double().cpu()
        assert float((got - ref).abs().max() / ref.abs().max()) <= TOL_POOLED


# ---------------------------------------------------------------------------------------------------------------------------
# b-d. each phase on its own inputs, the chain against the oracle, at the edges
# ---------------------------------------------------------------------------------------------------------------------------
TI, DJ = torch.tensor([0, 0, 1, 2, 2, 0]), torch.tensor([0, 1, 2, 1, 0, 1])     # equal indices on both sides, a duplicate pair


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("N", [1, 2, 31, 96, 127, 128, 129, 255, 256, 257, 640, 1024])
def test_phases_and_chain(N, mode):
    """point counts from a single point to the 1024-point Waymo config: full, ragged and single tiles"""
    m, orc = _pair()
    fmt = FMTS[mode]
    ot, od = _objects(3, N, N), _objects(3, N, N + 1)
    fx, pt, pd, dbg, L = _run(m, fmt, ot, od, TI, DJ)
    check_phases(fx, pt, pd, TI, DJ, dbg, f"{mode} N={N}")
    check_oracle(fx, orc, ot, od, TI, DJ, dbg, L, f"{mode} N={N}")


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("kind", ["same", "zero"])
@pytest.mark.parametrize("N", [1, 129, 256])
def test_degenerate_objects(N, kind, mode):
    """objects whose points are all identical, and all-zero features (empty crops), matched against ordinary objects and
    against each other"""
    m, orc = _pair()
    fmt = FMTS[mode]
    ot = _objects(3, N, 40 + N, kind=kind)
    od = _objects(3, N, 41 + N)
    od = (torch.cat([od[0][:2], ot[0][:1]]), torch.cat([od[1][:2], ot[1][:1]]))
    fx, pt, pd, dbg, L = _run(m, fmt, ot, od, TI, DJ)
    check_phases(fx, pt, pd, TI, DJ, dbg, f"{mode} {kind} N={N}")
    check_oracle(fx, orc, ot, od, TI, DJ, dbg, L, f"{mode} {kind} N={N}")


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("N", [1, 198, 256])
def test_token_sets(N, mode):
    """token sets without coordinates (ImageReIDNet's cross_lin_attn): no position code, PV = 0"""
    m, orc = _pair("image")
    fmt = FMTS[mode]
    ot, od = _objects(3, N, 60 + N, xyz=False), _objects(3, N, 61 + N, xyz=False)
    fx, pt, pd, dbg, L = _run(m, fmt, ot, od, TI, DJ)
    assert (_rows(pt.PV, fmt) == 0).all()
    check_phases(fx, pt, pd, TI, DJ, dbg, f"{mode} tokens N={N}")
    check_oracle(fx, orc, ot, od, TI, DJ, dbg, L, f"{mode} tokens N={N}")


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("scale", [1 / 16, 1 / 4, 1, 4, 16])
def test_feature_magnitude_sweep(scale, mode):
    """h scaled by 1/16 ... 16 around the encoder's range (max|h| ~ 2): every phase stays on the reference and the logits stay
    inside the mode's gate against the oracle (models/fused_pairs.py states the range)"""
    m, orc = _pair()
    fmt = FMTS[mode]
    ot, od = _objects(3, 256, 80, scale=scale), _objects(3, 256, 81, scale=scale)
    fx, pt, pd, dbg, L = _run(m, fmt, ot, od, TI, DJ)
    check_phases(fx, pt, pd, TI, DJ, dbg, f"{mode} x{scale}")
    check_oracle(fx, orc, ot, od, TI, DJ, dbg, L, f"{mode} x{scale}", logit_tol=GATE[fmt])


# ---------------------------------------------------------------------------------------------------------------------------
# e. scheduling: the persistent loops with many units per CTA, dense / duplicate / self / unsorted unit lists
# ---------------------------------------------------------------------------------------------------------------------------
def _outputs(dbg, L):
    return dict(A=dbg["A"], B7=dbg["B7"], part=dbg["part"], pooled=dbg["pooled"][0].t(), L=L)


def _assert_same(a, b, what):
    for k in a:
        assert torch.equal(a[k], b[k]), f"{what}: {k} differs"


@pytest.mark.parametrize("mode", ["parity_tc", "fast"])
@pytest.mark.parametrize("n_ctas", [1, 2])
def test_unit_scheduling_is_bit_exact(n_ctas, mode):
    """A CTA runs three groups over contiguous unit ranges; with 1 or 2 CTAs every group walks many units (template switches in
    phase 1a, cross-unit prefetch in phases 1b and 2).  Each unit's sums run in a fixed order whatever unit precedes it, so the
    results equal the default grid bit for bit, for the dense row block (r0 > 0), a pair list with duplicates and self-pairs on one
    set (pt is pd), and the same pairs unsorted."""
    m, _ = _pair()
    fmt, N = FMTS[mode], 200
    ot, od = _objects(7, N, 90), _objects(5, N, 91)
    r0, nrows, Dn = 2, 4, 5
    u = torch.arange(nrows * Dn)
    ti, dj = r0 + u // Dn, u % Dn
    _, _, _, dbg, L = _run(m, fmt, ot, od, ti, dj)
    ref = _outputs(dbg, L)
    for nc in (None, n_ctas):
        _, _, _, dbg, L = _run(m, fmt, ot, od, None, None, n_ctas=nc, dense=(r0, nrows, Dn))
        _assert_same(_outputs(dbg, L), ref, f"dense n_ctas={nc}")
        _, _, _, dbg, L = _run(m, fmt, ot, od, ti, dj, n_ctas=nc)
        _assert_same(_outputs(dbg, L), ref, f"pair list n_ctas={nc}")
    perm = torch.randperm(u.numel(), generator=torch.Generator().manual_seed(0))
    _, _, _, dbg, L = _run(m, fmt, ot, od, ti[perm], dj[perm], n_ctas=n_ctas)
    _assert_same(_outputs(dbg, L), {k: v[perm.to(v.device)] for k, v in ref.items()}, "unsorted")
    # one set against itself: (i, j) and (j, i) are the same two units with the roles swapped, (i, i) has equal roles
    ti = torch.tensor([3, 0, 6, 3, 2, 2, 5, 0, 3, 1, 6])
    dj = torch.tensor([3, 6, 0, 1, 2, 2, 4, 0, 3, 3, 0])
    fx, pt, pd, dbg, L = _run(m, fmt, ot, None, ti, dj, n_ctas=n_ctas)
    fx0, _, _, dbg0, L0 = _run(m, fmt, ot, None, ti, dj)
    _assert_same(_outputs(dbg, L), _outputs(dbg0, L0), "self pairs")
    for p in range(ti.numel()):
        for q in range(ti.numel()):
            if (ti[p], dj[p]) == (dj[q], ti[q]):
                assert torch.equal(dbg["A"][p, 0], dbg["A"][q, 1]) and torch.equal(dbg["part"][p, 0], dbg["part"][q, 1])
                assert torch.equal(L[p], L[q])
    check_phases(fx, pt, pd, ti, dj, dbg, f"{mode} self pairs n_ctas={n_ctas}")
