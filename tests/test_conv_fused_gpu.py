"""The trainer's tcgen05 conv kernels, one launch at a time, against a float64 reference.

Every convolution of a training step runs on one of five kernels -- the basic kernel with one or two MMA streams
(`nacc`), each with or without the staged-tile epilogue (`ms`: 1 = GroupNorm statistics on the tensor core, 2 = TMA
store only), and the persistent row-tile kernel (resident or streamed weights) -- with the shared epilogue of
csrc/epilogue.cuh: bias, second bias, per-image row, residual, pitched outputs, and the two fused GroupNorm hooks
(statistics of the stored output; gn-bwd: dz = dy * act'(z) in place of dy plus the sums of dz and dz * xhat).  The
weight gradients run in accumulate mode (TMA reduce-add, fused bias gradients, finalize for 3x3).  Each case here goes
through ub_conv2d_nhwc_fused / ub_conv2d_nhwc_wgrad_acc and asserts the plan it means to cover (UbConvPlanInfo), so a
planner change cannot silently move it onto another kernel.

References: float64 torch on the CPU, on the same bf16-rounded operands; weights are packed by ub_pack_conv_weight
(dgrad cases use the `wd` pack and conv_transpose2d, which pins the pack too).  With A = the same sums over absolute
values (conv(|x|, |w|) + |addends|), per element:
  * bf16 outputs : |got - ref| <= 2^-8 |ref| + 1e-4 A      (round to nearest bf16 + fp32 accumulation)
  * fp32 outputs : |got - ref| <= 1e-4 A
  * statistics   : against the kernel's own stored bf16 output (float64 sums): 1e-5 of sum |y| and of sum y^2 per
                   (image, channel); and what GroupNorm consumes, the per-(image, group) variance, within 1e-3 relative
                   (a 4-sigma channel offset is among the cases).  The tensor-core statistics (ms == 1) take the sum of
                   squares from the diagonal of the Gram matrix Y^T Y, every y^2 exact, so the tight bound holds there
                   too, at BN 64 and 128 with one or two images per tile (with a staged bf16(y^2) operand the
                   variance was off by 7.3e-3 at 32x32 and 6.8e-3 at 8x8 with the 4-sigma offset, and the sum of
                   squares by 39x and 85x the 1e-5 bound).
  * gn-bwd dz    : against f * s (1 + z (1 - s)) in float64 (the value the stored bf16 rounds), s = sigmoid(z), f =
                   the float64 conv output plus addend, z = gamma * xhat + beta from the statistics passed in (eps 1e-5):
                   |got - ref| <= 2^-8 |ref| + (1 + 2^-8) (|act'(z)| 1e-4 A + |f| 2^-11.9 (1 + |z|)).
                   The last term is the kernel's sigmoid, 0.5 + 0.5 tanh.approx(z / 2): tanh.approx has a relative error
                   below 2^-10.99, so s is off by at most 2^-11.99 and act'(z) = s (1 + z - z s) by at most that times
                   |d act' / ds| = |1 + z - 2 z s| <= 1 + |z| (2^-11.9 leaves room for the fp32 z).
  * gn-bwd S     : against the stored dz and float64 xhat: 1e-5 of sum |dz| and of sum |dz * xhat|.
Sentinels pin what is written: outputs (pitch padding, the other channels of a concat buffer and a guard region
included) start as NaN; stats, S, dbias and a 1x1 dweight start at known non-zero values -- every target element must
be written, nothing else may change, accumulators must add to their start value.

At B = 32 the conv reference covers images 0, 1, 2, B/2, B-2 and B-1 (the first and last tiles included, >= 20000
elements); the statistics, S and the finite / untouched checks cover every image.
"""
import ctypes as C
import os

import pytest
import torch
import torch.nn.functional as F

from gpu_util import TOL_BF16

pytestmark = pytest.mark.gpu

U = 2.0 ** -8         # bf16 unit roundoff (round to nearest)
EPS_ACC = 1e-4        # fp32 accumulation, of A
EPS_SUM = 1e-5        # the hooks' fp32 sums, of the sum of absolute values
TANH = 2.0 ** -11.9   # the hook's sigmoid (tanh.approx), see the module docstring
GUARD = 4096          # elements behind every output that must stay untouched
G = 32                # GroupNorm groups


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _rnd(g, *shape, scale=1.0, shift=0.0):
    return torch.randn(*shape, generator=g, dtype=torch.float64) * scale + shift


def _bf(t):
    """float64 tensor rounded to bf16 values (kept in float64)."""
    return t.to(torch.bfloat16).double()


def _pitched(x, ld):
    """NHWC bf16 device copy of x (float64, bf16 values) with channel pitch ld; the padding holds NaN."""
    B, H, W, Cc = x.shape
    buf = torch.full((B, H, W, ld), -1, dtype=torch.int16).view(torch.bfloat16)
    buf[..., :Cc] = x.to(torch.bfloat16)
    return buf.cuda()


def _conv(x, w, k, dgrad):
    """float64 NHWC -> NHWC: fprop conv2d with w (Cout, Cin, k, k), or dgrad = conv_transpose2d with the layer weight
    w (C_dy, C_dx, k, k)."""
    xn = x.permute(0, 3, 1, 2)
    y = F.conv_transpose2d(xn, w, padding=k // 2) if dgrad else F.conv2d(xn, w, padding=k // 2)
    return y.permute(0, 2, 3, 1)


def _sample(B):
    return list(range(B)) if B <= 8 else sorted({0, 1, 2, B // 2, B - 2, B - 1})


def _group_stats(s, ss, n):
    """per-(image, group) mean and variance from per-(image, channel) sums [B][C] over n = HW pixels"""
    B, Cc = s.shape
    cpg = Cc // G
    sg, ssg = s.reshape(B, G, cpg).sum(-1), ss.reshape(B, G, cpg).sum(-1)
    mean = sg / (cpg * n)
    return mean, ssg / (cpg * n) - mean * mean


# ------------------------------------------------------------------------------------------------ conv cases
# segs: (C_in, ldx, ksize, dgrad).  A dgrad segment reads dy (C_in channels) with the wd pack of a layer whose input has
# C_out channels.  ep: bias / bias2 / rowvec / residual (= ldr) / stats / gn (= gn silu) / ldo / out_mode / offset
# (added to the bias: a channel offset for the variance check) / gn_ldx.  expect: UbConvPlanInfo fields.
def case(name, kernel, B, H, W, Cout, segs, expect, **ep):
    return pytest.param(dict(name=name, kernel=kernel, B=B, H=H, W=W, Cout=Cout, segs=segs, expect=expect, ep=ep),
                        id=name)


CONV_CASES = [
    # basic kernel, two MMA streams, per-thread epilogue: a 120-pixel (ragged) tile, 4 CTAs
    case("basic_nacc2_ms0_ragged", 0, 2, 12, 20, 64, [(64, 64, 3, False)], dict(nacc=2, ms=0, TB=1),
         bias=1, rowvec=1, residual=96, stats=1),
    # basic, one stream (256 CTAs), tensor-core statistics / staged TMA store
    case("basic_nacc1_ms1_stats", 0, 32, 32, 32, 64, [(64, 64, 3, False)], dict(nacc=1, ms=1, BN=64, TB=1),
         bias=1, stats=1, offset=4.0),
    case("basic_nacc1_ms2_plain", 0, 32, 32, 32, 64, [(64, 64, 3, False)], dict(nacc=1, ms=2, BN=64)),
    # tensor-core statistics at BN 128 (M = 128, the Gram matrix spans two 64-channel atoms): the 32x32 level's
    # stats-hooked convs of the default model
    case("basic_nacc1_ms1_bn128", 0, 32, 32, 32, 128, [(128, 128, 3, False)], dict(nacc=1, ms=1, BN=128, TB=1),
         bias=1, stats=1, offset=4.0),
    # basic, two images per tile with an odd batch (the last tile is half empty), tensor-core statistics, a 4-sigma
    # channel offset, and the per-image rows of both images staged
    case("basic_ms1_tb2_oddB_offset", 0, 5, 8, 8, 128, [(128, 128, 3, False)], dict(nacc=2, ms=1, BN=64, TB=2),
         bias=1, rowvec=1, stats=1, offset=4.0),
    # the same at BN 128 (128 two-image tiles, the last one half empty): one Gram matrix per image
    case("basic_ms1_tb2_oddB_bn128", 0, 255, 8, 8, 128, [(128, 128, 3, False)], dict(nacc=2, ms=1, BN=128, TB=2),
         bias=1, rowvec=1, stats=1, offset=4.0),
    # the same with an N tile the tensor-core statistics do not take (BN 96): shuffle statistics of a two-image tile
    case("basic_ms0_tb2_oddB_bn96", 0, 3, 8, 8, 96, [(64, 64, 3, False)], dict(nacc=2, ms=0, BN=96, TB=2),
         rowvec=1, stats=1),
    # basic, staged TMA store into a wider (concat) buffer, bias + bias2
    case("basic_nacc2_ms2_concat", 0, 2, 16, 16, 128, [(128, 128, 3, False)], dict(nacc=2, ms=2, BN=64),
         bias=1, bias2=1, ldo=192),
    # basic, 3x3 + 1x1 skip conv (both inputs pitched) with the second bias, statistics at the 384-channel width
    case("basic_two_segments", 0, 2, 16, 16, 384, [(64, 128, 3, False), (192, 256, 1, False)],
         dict(nacc=2, ms=1, BN=64, TB=1),
         bias=1, bias2=1, stats=1),
    # basic, fp32 outputs (the drop-in layer operators' path)
    case("basic_nhwc_f32", 0, 32, 32, 32, 64, [(64, 64, 3, False)], dict(nacc=1, ms=0, BN=64),
         bias=1, rowvec=1, out_mode=2, ldo=68),
    case("basic_nchw_f32", 0, 3, 13, 11, 96, [(64, 64, 3, False)], dict(nacc=2, ms=0, BN=96),
         bias=1, rowvec=1, out_mode=1),
    # basic, gn-bwd hook on dgrads (wd pack), GroupNorm input pitched; 2, 6, 10, 12 and 14 channels per group: the
    # non-power-of-two groups straddle the 64-channel N tiles
    case("basic_gnbwd_c64_silu1", 0, 2, 16, 16, 64, [(128, 128, 3, True)], dict(nacc=2, ms=0, BN=64), gn=1, gn_ldx=72),
    case("basic_gnbwd_c192_silu0", 0, 2, 16, 16, 192, [(128, 128, 3, True)], dict(nacc=2, ms=0, BN=64), gn=0, gn_ldx=256),
    case("basic_gnbwd_c320_silu1", 0, 2, 16, 16, 320, [(128, 128, 3, True)], dict(nacc=2, ms=0, BN=64), gn=1, gn_ldx=328),
    case("basic_gnbwd_c384_silu1", 0, 3, 8, 8, 384, [(128, 128, 3, True)], dict(nacc=2, ms=0, BN=64, TB=2), gn=1, gn_ldx=392),
    case("basic_gnbwd_c448_silu1", 0, 2, 16, 16, 448, [(128, 136, 1, True)], dict(nacc=1, ms=0, BN=64), gn=1, gn_ldx=512),
    # row-tile kernel, resident weights (one segment, C_in <= 64, one N tile)
    case("rows_resident_stats", 1, 2, 64, 64, 64, [(64, 64, 3, False)], dict(kernel=1, w_resident=1, BN=64),
         bias=1, stats=1),
    case("rows_resident_persistent", 1, 32, 64, 64, 64, [(64, 64, 3, False)], dict(kernel=1, w_resident=1, BN=64, grid=148),
         bias=1, rowvec=1, stats=1),
    # row-tile, streamed weights, persistent loop (512 tiles on 148 CTAs), gn-bwd hook with SiLU
    case("rows_streamed_gnbwd", 1, 32, 64, 64, 64, [(192, 192, 3, True)], dict(kernel=1, w_resident=0, BN=64, grid=148),
         gn=1, gn_ldx=128),
    # row-tile, partial last tile (W 16: 16-row tiles, H 24), C_in not a multiple of 64, residual + statistics
    case("rows_partial_tile", 1, 3, 24, 16, 64, [(96, 104, 3, False)], dict(kernel=1, w_resident=0, BN=64, TH=16),
         residual=64, stats=1),
    # row-tile, 3x3 + 1x1 skip conv, bias2, statistics at the 192-channel width (BN 96)
    case("rows_two_segments", 1, 2, 32, 32, 192, [(128, 128, 3, False), (64, 64, 1, False)],
         dict(kernel=1, w_resident=0, BN=96), bias=1, bias2=1, stats=1),
]

STATS0 = (0.75, 1.5)   # start values of stats / gn_S (sum, second sum)


def _setup(cs, seed):
    """Host operands (float64, bf16 values) and device buffers of one case."""
    g = torch.Generator().manual_seed(seed)
    B, H, W, Cout, ep = cs["B"], cs["H"], cs["W"], cs["Cout"], cs["ep"]
    h = dict(segs=[])
    d = dict(keep=[])
    for (cin, ldx, k, dgrad) in cs["segs"]:
        x = _bf(_rnd(g, B, H, W, cin))
        # layer weight: fprop (Cout, cin, k, k); dgrad (cin, Cout, k, k), i.e. dy has cin channels
        w = _bf(_rnd(g, *((cin, Cout) if dgrad else (Cout, cin)), k, k, scale=(cin * k * k) ** -0.5))
        h["segs"].append((x, w, k, dgrad))
        xd = _pitched(x, ldx)
        wp = torch.empty(k * k * cin * Cout, dtype=torch.bfloat16, device="cuda")
        wdev = w.float().cuda()
        # ub_pack_conv_weight(weight, wf, wd, C_in, C_out, ksize) of the layer
        if dgrad:
            rc = _lib().ub_pack_conv_weight(_p(wdev), None, _p(wp), Cout, cin, k)
        else:
            rc = _lib().ub_pack_conv_weight(_p(wdev), _p(wp), None, cin, Cout, k)
        assert rc == 0, _lib().ub_last_error()
        d["keep"] += [xd, wp, wdev]
        d.setdefault("segs", []).append((xd, cin, ldx, wp, k))
    off = ep.get("offset", 0.0)
    for nm in ("bias", "bias2"):
        if ep.get(nm):
            h[nm] = _rnd(g, Cout, scale=0.5, shift=off if nm == "bias" else 0.0).float().double()
            d[nm] = h[nm].float().cuda()
    if ep.get("rowvec"):
        h["rowvec"] = _rnd(g, B, Cout, scale=0.5).float().double()
        d["rowvec"] = h["rowvec"].float().cuda()
    if ep.get("residual"):
        h["residual"] = _bf(_rnd(g, B, H, W, Cout))
        d["residual"] = _pitched(h["residual"], ep["residual"])
    if ep.get("stats"):
        st = torch.empty(B, Cout, 2)
        st[..., 0], st[..., 1] = STATS0
        d["stats"] = st.cuda()
    if "gn" in ep:
        gx = _bf(_rnd(g, B, H, W, Cout, scale=1.3, shift=0.2))
        h["gn_x"] = gx
        cs_ = torch.stack([gx.sum((1, 2)), (gx * gx).sum((1, 2))], -1)   # [B][C][2], float64
        h["chsum"] = cs_.float().double()
        h["gamma"] = (1.0 + 0.3 * _rnd(g, Cout)).float().double()
        h["beta"] = (0.2 * _rnd(g, Cout)).float().double()
        d["gn_x"] = _pitched(gx, ep["gn_ldx"])
        d["chsum"], d["gamma"], d["beta"] = (h[k].float().cuda() for k in ("chsum", "gamma", "beta"))
        S = torch.empty(B, Cout, 2)
        S[..., 0], S[..., 1] = STATS0
        d["S"] = S.cuda()
    mode = ep.get("out_mode", 0)
    ldo = ep.get("ldo", Cout)
    if mode == 0:
        d["out"] = torch.full((B * H * W * ldo + GUARD,), -1, dtype=torch.int16).view(torch.bfloat16).cuda()
    elif mode == 2:
        d["out"] = torch.full((B * H * W * ldo + GUARD,), float("nan")).cuda()
    else:
        d["out"] = torch.full((B * Cout * H * W + GUARD,), float("nan")).cuda()
    return h, d


def _lib():
    import __graft_entry__ as ge
    return ge.load_package().lib()


def _launch(cs, d):
    """ub_conv2d_nhwc_fused; returns (rc, UbConvPlanInfo)."""
    import __graft_entry__ as ge
    ub = ge.load_package()
    ep = cs["ep"]
    segs = (ub.UbConvSeg * 2)()
    for i, (xd, cin, ldx, wp, k) in enumerate(d["segs"]):
        segs[i] = ub.UbConvSeg(_p(xd), cin, ldx, _p(wp), k)
    e = ub.UbConvEpilogue()
    e.bias, e.bias2, e.rowvec = _p(d.get("bias")), _p(d.get("bias2")), _p(d.get("rowvec"))
    e.residual_bf16, e.ldr = _p(d.get("residual")), ep.get("residual", 0)
    e.out, e.ldo, e.out_mode = _p(d["out"]), ep.get("ldo", 0), ep.get("out_mode", 0)
    e.stats = _p(d.get("stats"))
    if "gn" in ep:
        e.gn_x_bf16, e.gn_ldx = _p(d["gn_x"]), ep["gn_ldx"]
        e.gn_chsum, e.gn_gamma, e.gn_beta, e.gn_S = _p(d["chsum"]), _p(d["gamma"]), _p(d["beta"]), _p(d["S"])
        e.gn_silu, e.gn_groups = ep["gn"], G
    info = ub.UbConvPlanInfo()
    rc = ub.lib().ub_conv2d_nhwc_fused(segs, len(d["segs"]), cs["B"], cs["H"], cs["W"], cs["Cout"], C.byref(e),
                                       cs["kernel"], C.byref(info))
    torch.cuda.synchronize()
    return rc, info


PLAN_KEYS = ("kernel", "BN", "nacc", "ms", "stages", "w_resident", "TW", "TH", "TB", "grid")


def _plan(info):
    return {k: getattr(info, k) for k in PLAN_KEYS}


def _assert_plan(cs, info):
    plan = _plan(info)
    want = {"kernel": cs["kernel"], **cs["expect"]}
    assert all(plan[k] == v for k, v in want.items()), (cs["name"], plan, want)
    return plan


def _worst(err, bound):
    return float((err / bound).max())


def _check_gn(cs, h, y_all, conv, A):
    """gn-bwd hook: dz per element (sampled images), S (every image).  Returns the worst error / bound ratios."""
    B, H, W, Cout = cs["B"], cs["H"], cs["W"], cs["Cout"]
    silu = cs["ep"]["gn"]
    mean, var = _group_stats(h["chsum"][..., 0], h["chsum"][..., 1], H * W)   # what the kernel derives, in float64
    cpg = Cout // G
    rstd = (var + 1e-5).rsqrt()
    mean_c, rstd_c = mean.repeat_interleave(cpg, 1), rstd.repeat_interleave(cpg, 1)   # [B][C]
    xhat = (h["gn_x"] - mean_c[:, None, None, :]) * rstd_c[:, None, None, :]
    out = {}
    if conv is not None:
        imgs, f = conv
        z = h["gamma"] * xhat[imgs] + h["beta"]
        if silu:
            s = torch.sigmoid(z)
            act = s * (1 + z * (1 - s))
        else:
            act = torch.ones_like(z)
        ref = f * act
        bound = U * ref.abs() + (1 + U) * (act.abs() * EPS_ACC * A + (f.abs() * TANH * (1 + z.abs()) if silu else 0))
        out["dz"] = _worst((y_all[imgs] - ref).abs(), bound)
        assert out["dz"] <= 1.0, (cs["name"], "dz", out["dz"])
    S = h["S_got"] - torch.tensor(STATS0, dtype=torch.float64)
    p = y_all * xhat
    S_ref = torch.stack([y_all.sum((1, 2)), p.sum((1, 2))], -1)
    S_abs = torch.stack([y_all.abs().sum((1, 2)), p.abs().sum((1, 2))], -1)
    out["S"] = _worst((S - S_ref).abs(), EPS_SUM * S_abs + 1e-30)
    assert out["S"] <= 1.0, (cs["name"], "S", out["S"])
    return out


def _check_stats(cs, st_got, y_all):
    """statistics hook against the stored bf16 output (every image): the sums, then the group variance GroupNorm
    derives from them.  Returns the worst ratios."""
    HW = cs["H"] * cs["W"]
    st = st_got - torch.tensor(STATS0, dtype=torch.float64)
    s_ref, ss_ref = y_all.sum((1, 2)), (y_all * y_all).sum((1, 2))
    out = {}
    m_got, v_got = _group_stats(st[..., 0], st[..., 1], HW)
    m_ref, v_ref = _group_stats(s_ref, ss_ref, HW)
    out["var_rel"] = float(((v_got - v_ref).abs() / v_ref).max())
    out["mean_rstd"] = float(((m_got - m_ref).abs() / v_ref.sqrt()).max())
    out["sum"] = _worst((st[..., 0] - s_ref).abs(), EPS_SUM * y_all.abs().sum((1, 2)) + 1e-30)
    out["sumsq"] = _worst((st[..., 1] - ss_ref).abs(), EPS_SUM * ss_ref + 1e-30)
    print(f"    stats: variance rel err {out['var_rel']:.2e} (bound 1e-3), mean err / std {out['mean_rstd']:.2e}")
    assert out["var_rel"] <= 1e-3 and out["mean_rstd"] <= 1e-4, (cs["name"], out)
    assert out["sum"] <= 1.0 and out["sumsq"] <= 1.0, (cs["name"], out)
    return out


@pytest.mark.parametrize("cs", CONV_CASES)
def test_conv_fused(ub, cs):
    torch.set_num_threads(os.cpu_count() or 1)
    B, H, W, Cout, ep = cs["B"], cs["H"], cs["W"], cs["Cout"], cs["ep"]
    h, d = _setup(cs, seed=sum(map(ord, cs["name"])))
    n0 = ub.lib().ub_launch_count()
    rc, info = _launch(cs, d)
    assert rc == 0, ub.lib().ub_last_error()
    assert ub.lib().ub_launch_count() == n0 + 1
    plan = _assert_plan(cs, info)
    mode, ldo = ep.get("out_mode", 0), ep.get("ldo", Cout)

    # what was written: every target element, and nothing else
    out = d["out"].cpu()
    npix = B * H * W
    if mode == 0:
        bits = out.view(torch.int16)
        body = out[:npix * ldo].reshape(B, H, W, ldo)
        assert bool((bits[:npix * ldo].reshape(B, H, W, ldo)[..., Cout:] == -1).all()), "wrote outside [0, C_out)"
        assert bool((bits[npix * ldo:] == -1).all()), "wrote past the output"
        y_all = body[..., :Cout].double()
    elif mode == 2:
        body = out[:npix * ldo].reshape(B, H, W, ldo)
        assert bool(body[..., Cout:].isnan().all()) and bool(out[npix * ldo:].isnan().all()), "wrote outside"
        y_all = body[..., :Cout].double()
    else:
        assert bool(out[npix * Cout:].isnan().all()), "wrote past the output"
        y_all = out[:npix * Cout].reshape(B, Cout, H, W).permute(0, 2, 3, 1).double()
    assert bool(y_all.isfinite().all()), "an output element was not written"

    # float64 reference on the sampled images
    imgs = _sample(B)
    f = torch.zeros(len(imgs), H, W, Cout, dtype=torch.float64)
    A = torch.zeros_like(f)
    for (x, w, k, dgrad) in h["segs"]:
        f += _conv(x[imgs], w, k, dgrad)
        A += _conv(x[imgs].abs(), w.abs(), k, dgrad)
    for nm in ("bias", "bias2"):
        if nm in h:
            f += h[nm]
            A += h[nm].abs()
    if "rowvec" in h:
        f += h["rowvec"][imgs][:, None, None, :]
        A += h["rowvec"][imgs].abs()[:, None, None, :]
    if "residual" in h:
        f += h["residual"][imgs]
        A += h["residual"][imgs].abs()

    res = {}
    if "gn" in ep:
        h["S_got"] = d["S"].cpu().double()
        res = _check_gn(cs, h, y_all, (imgs, f), A)
    else:
        got = y_all[imgs]
        bound = (U * f.abs() + EPS_ACC * A) if mode == 0 else EPS_ACC * A
        res["out"] = _worst((got - f).abs(), bound)
        assert res["out"] <= 1.0, (cs["name"], "out", res["out"])
    if ep.get("stats"):
        res.update(_check_stats(cs, d["stats"].cpu().double(), y_all))
    print(f"[{cs['name']}] plan " + " ".join(f"{k}={plan[k]}" for k in ("kernel", "BN", "nacc", "ms", "TB",
                                                                         "w_resident", "grid")) +
          "  worst error / bound: " + " ".join(f"{k}={v:.3f}" for k, v in res.items() if k not in ("var_rel",
                                                                                                     "mean_rstd")))


# ------------------------------------------------------------------------------------------------ weight gradients
#              name        B   H   W  Cin Cout k  lddy  ldx  bias bias2 expect
WGRAD_CASES = [
    pytest.param("col3x3", 3, 16, 16, 128, 64, 3, 128, 192, 1, 1, dict(colmode=1), id="col3x3"),
    pytest.param("row3x3", 4, 4, 4, 64, 128, 3, 192, 64, 1, 0, dict(colmode=0), id="row3x3"),
    pytest.param("k1x1", 2, 32, 32, 192, 64, 1, 64, 256, 1, 1, dict(colmode=0), id="k1x1"),
    pytest.param("split3x3", 32, 32, 32, 64, 64, 3, 64, 64, 1, 0, dict(colmode=1, split=True), id="split3x3"),
]


def _wgrad_setup(B, H, W, Cin, Cout, lddy, ldx, seed):
    g = torch.Generator().manual_seed(seed)
    dy = _bf(_rnd(g, B, H, W, Cout))
    x = _bf(_rnd(g, B, H, W, Cin))
    return dy, x, _pitched(dy, lddy), _pitched(x, ldx)


def _wgrad_call(ub, dyd, lddy, xd, ldx, dw, db, db2, B, H, W, Cin, Cout, k):
    colmode, nsplit = C.c_int(-1), C.c_int(-1)
    n0 = ub.lib().ub_launch_count()
    rc = ub.lib().ub_conv2d_nhwc_wgrad_acc(_p(dyd), lddy, _p(xd), ldx, _p(dw), _p(db), _p(db2), B, H, W, Cin, Cout, k,
                                           C.byref(colmode), C.byref(nsplit))
    torch.cuda.synchronize()
    assert rc == 0, ub.lib().ub_last_error()
    assert ub.lib().ub_launch_count() == n0 + (2 if k == 3 else 1)
    return colmode.value, nsplit.value


@pytest.mark.parametrize("name,B,H,W,Cin,Cout,k,lddy,ldx,bias,bias2,expect", WGRAD_CASES)
def test_wgrad_acc(ub, name, B, H, W, Cin, Cout, k, lddy, ldx, bias, bias2, expect):
    """Accumulate-mode weight gradient: 3x3 dweight overwritten through the zeroed workspace (NaN start), 1x1 dweight,
    dbias and dbias2 added to their start values; run twice -- the finalize must leave the workspace zeroed, so both
    runs agree up to the order of the fp32 reductions."""
    torch.set_num_threads(os.cpu_count() or 1)
    dy, x, dyd, xd = _wgrad_setup(B, H, W, Cin, Cout, lddy, ldx, seed=len(name) + B)
    xn, dyn = x.permute(0, 3, 1, 2), dy.permute(0, 3, 1, 2)
    dw_ref = torch.nn.grad.conv2d_weight(xn, (Cout, Cin, k, k), dyn, padding=k // 2)
    A_w = torch.nn.grad.conv2d_weight(xn.abs(), (Cout, Cin, k, k), dyn.abs(), padding=k // 2)
    db_ref, A_b = dy.sum((0, 1, 2)), dy.abs().sum((0, 1, 2))
    W0, B0, B20 = (float("nan") if k == 3 else 0.5), 0.25, -0.5
    runs = []
    for _ in range(2):
        dw = torch.full((Cout, Cin, k, k), W0, device="cuda")
        db = torch.full((Cout,), B0, device="cuda") if bias else None
        db2 = torch.full((Cout,), B20, device="cuda") if bias2 else None
        colmode, nsplit = _wgrad_call(ub, dyd, lddy, xd, ldx, dw, db, db2, B, H, W, Cin, Cout, k)
        assert colmode == expect["colmode"], (colmode, nsplit)
        if expect.get("split"):
            assert nsplit > 1, nsplit
        got = dw.cpu().double() - (0.0 if k == 3 else W0)
        worst = {"dw": _worst((got - dw_ref).abs(), EPS_ACC * A_w + 1e-30)}
        if bias:
            worst["db"] = _worst((db.cpu().double() - B0 - db_ref).abs(), EPS_ACC * A_b + 1e-30)
        if bias2:
            worst["db2"] = _worst((db2.cpu().double() - B20 - db_ref).abs(), EPS_ACC * A_b + 1e-30)
        assert all(v <= 1.0 for v in worst.values()), (name, worst)
        runs.append(got)
    agree = _worst((runs[1] - runs[0]).abs(), 1e-5 * A_w + 1e-30)
    assert agree <= 1.0, ("second run differs", agree)
    print(f"[wgrad {name}] plan colmode={colmode} nsplit={nsplit}  worst error / bound: "
          + " ".join(f"{k_}={v:.3f}" for k_, v in worst.items()) + f" run2-run1={agree:.3f}")


# ------------------------------------------------------------------------------------------------ GroupNorm chain
@pytest.mark.parametrize("Cc,silu,add", [(64, 1, False), (192, 1, True), (320, 0, True)])
def test_gnbwd_hook_then_apply(ub, Cc, silu, add):
    """A ResBlock's GroupNorm(+SiLU) backward as the trainer runs it: the dgrad conv that produces dL/d act(gn(x))
    with the gn-bwd hook, then ub_groupnorm_nhwc_backward_apply (with and without the residual-gradient input) --
    against float64 autograd of GroupNorm + SiLU with the float64 conv output as the upstream gradient.  Bounds of
    test_groupnorm_nhwc_gpu.py: dx within 2e-2 of its max and 1e-2 relative L2; dgamma, dbeta 1e-2 relative L2."""
    torch.set_num_threads(os.cpu_count() or 1)
    B, H, W, Cdy = 2, 16, 16, 128
    cs = dict(name=f"chain_c{Cc}", kernel=0, B=B, H=H, W=W, Cout=Cc, segs=[(Cdy, Cdy, 3, True)],
              expect=dict(nacc=2, ms=0, BN=64, TB=1),
              ep=dict(gn=silu, gn_ldx=Cc))
    h, d = _setup(cs, seed=Cc + silu)
    d["S"].zero_()   # the apply pass consumes S: it starts at zero, as in the trainer
    rc, info = _launch(cs, d)
    assert rc == 0, ub.lib().ub_last_error()
    _assert_plan(cs, info)
    g = torch.Generator().manual_seed(7)
    addt = _bf(_rnd(g, B, H, W, Cc)) if add else None
    add_d = addt.to(torch.bfloat16).cuda() if add else None
    x_d = h["gn_x"].to(torch.bfloat16).cuda()
    dx = torch.full((B, H, W, Cc), -1, dtype=torch.int16).view(torch.bfloat16).cuda()
    dgam, dbet = torch.full((Cc,), 0.5, device="cuda"), torch.full((Cc,), -0.25, device="cuda")
    rc = ub.lib().ub_groupnorm_nhwc_backward_apply(_p(x_d), _p(d["out"]), _p(d["chsum"]), _p(d["S"]), _p(d["gamma"]),
                                                   _p(d["beta"]), _p(add_d), _p(dx), _p(dgam), _p(dbet), B, H, W, Cc,
                                                   G, silu)
    torch.cuda.synchronize()
    assert rc == 0, ub.lib().ub_last_error()

    (x, w, k, dgrad), = h["segs"]
    f = _conv(x, w, k, dgrad).permute(0, 3, 1, 2)
    xr = h["gn_x"].permute(0, 3, 1, 2).clone().requires_grad_(True)
    gr, br = h["gamma"].clone().requires_grad_(True), h["beta"].clone().requires_grad_(True)
    z = F.group_norm(xr, G, gr, br, eps=1e-5)
    (F.silu(z) if silu else z).backward(f)
    dx_ref = xr.grad.permute(0, 2, 3, 1) + (addt if add else 0)
    got = dx.cpu().double()

    def rel_l2(a, b):
        return float((a - b).norm() / (b.norm() + 1e-30))

    r = {"dx_inf": float((got - dx_ref).abs().max() / dx_ref.abs().max()) / TOL_BF16,
         "dx_l2": rel_l2(got, dx_ref) / 1e-2,
         "dgamma": rel_l2(dgam.cpu().double() - 0.5, gr.grad) / 1e-2,
         "dbeta": rel_l2(dbet.cpu().double() + 0.25, br.grad) / 1e-2}
    print(f"[chain C={Cc} silu={silu} add={add}] plan BN={info.BN} nacc={info.nacc} ms={info.ms}  worst error / bound: "
          + " ".join(f"{k_}={v:.3f}" for k_, v in r.items()))
    assert all(v <= 1.0 for v in r.values()), r


# ------------------------------------------------------------------------------------------------ coverage, rejections
def test_case_matrix_covers_every_variant(ub):
    """The union of the cases' plans holds every kernel variant the trainer runs: basic nacc 1/2 x ms 0/1/2, two-image
    tiles with an odd batch, row-tile resident / streamed / partial last tile, both hooks on both kernels, and both
    3x3 weight-gradient modes plus the 1x1 one."""
    seen = set()
    for prm in CONV_CASES:
        cs = prm.values[0]
        _, d = _setup(cs, seed=1)
        rc, info = _launch(cs, d)
        assert rc == 0, (cs["name"], ub.lib().ub_last_error())
        p = _assert_plan(cs, info)
        ep = cs["ep"]
        hook = "stats" if ep.get("stats") else ("gn" if "gn" in ep else None)
        if p["kernel"] == 0:
            seen.add(("basic", p["nacc"], p["ms"]))
            if p["ms"] == 1:
                seen.add(("ms1", p["BN"], p["TB"]))
            if p["TB"] == 2 and cs["B"] % 2:
                seen.add(("tb2_odd_batch", p["ms"]))
        else:
            seen.add(("rows", "resident" if p["w_resident"] else "streamed"))
            if cs["H"] % p["TH"]:
                seen.add(("rows", "partial"))
        if hook:
            seen.add((hook, p["kernel"]))
    for prm in WGRAD_CASES:
        name, B, H, W, Cin, Cout, k, lddy, ldx, bias, bias2, _ = prm.values
        _, _, dyd, xd = _wgrad_setup(B, H, W, Cin, Cout, lddy, ldx, seed=1)
        dw = torch.zeros(Cout, Cin, k, k, device="cuda")
        colmode, nsplit = _wgrad_call(ub, dyd, lddy, xd, ldx, dw, None, None, B, H, W, Cin, Cout, k)
        seen.add(("wgrad", k, colmode))
        if nsplit > 1:
            seen.add(("wgrad", "split"))
    want = {("basic", n, m) for n in (1, 2) for m in (0, 1, 2)} | {("tb2_odd_batch", 0), ("tb2_odd_batch", 1)}
    want |= {("ms1", bn, tb) for bn in (64, 128) for tb in (1, 2)}   # M = 64 / 128 Gram layouts, one or two images
    want |= {("rows", "resident"), ("rows", "streamed"), ("rows", "partial")}
    want |= {("stats", 0), ("stats", 1), ("gn", 0), ("gn", 1)}
    want |= {("wgrad", 3, 1), ("wgrad", 3, 0), ("wgrad", 1, 0), ("wgrad", "split")}
    assert want <= seen, sorted(map(str, want - seen))


def test_conv_fused_rejects_unsupported(ub):
    """Unsupported requests return UB_ERR_SHAPE without launching anything: the row-tile kernel at an ineligible width,
    both hooks at once, a hook with an fp32 output, a bf16 output pitch that is not a multiple of 8 channels."""
    base = dict(name="reject", kernel=0, B=2, H=16, W=16, Cout=64, segs=[(64, 64, 3, False)], expect={}, ep={})
    bad = [
        dict(base, kernel=1, W=12, ep=dict(stats=1)),                                    # row-tile, W = 12
        dict(base, ep=dict(stats=1, gn=1, gn_ldx=64)),                                   # stats + gn_x
        dict(base, ep=dict(stats=1, out_mode=2)),                                        # hook, fp32 output
        dict(base, ep=dict(ldo=68)),                                                     # 136-byte pixel pitch
    ]
    L = ub.lib()
    for cs in bad:
        _, d = _setup(cs, seed=2)
        n0 = L.ub_launch_count()
        rc, info = _launch(cs, d)
        assert rc == -1, (cs["ep"], rc)
        assert L.ub_launch_count() == n0, cs["ep"]
        assert info.kernel == cs["kernel"]
        assert L.ub_last_error().decode()
