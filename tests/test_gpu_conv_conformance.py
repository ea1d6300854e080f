"""Conformance of the fused BatchNorm -> conv -> ReLU layers (csrc/conv.cu) in the regimes the
model runs them, and in the ones a rewrite of the persistent tile loop is most likely to break.

Compared with tests/test_gpu_kernels.py (max-norm errors at B <= 130, Gaussian inputs) these tests
  * run every layer, pass and conv precision mode at B = 1, 64, 1024 and at B_trip(l), a batch
    large enough that every CTA of a persistent kernel walks its tile loop at least twice (so the
    stage-ring parity flips and the last wave is ragged);
  * bound every output ELEMENT: |got - ref64| <= bar * S + floor, S = the same computation on
    absolute values, bar = max(tau(mode), 3 x the worst ratio of the same computation done by
    torch in float32 without TF32) -- an error confined to one tap, channel or tile edge cannot
    hide under the tensor's maximum;
  * feed ReLU-like inputs (half exact zeros, an all-zero channel, a channel with mean 100 and
    std 1) and gradients whose channels span 2^-20 .. 1;
  * place every output inside NaN guard bands and check that a kernel writes only what it owns,
    and that the ACCUMULATED / OVERWRITTEN contracts of include/ava_b200.h hold;
  * require bit-identical outputs when a batch is run in chunks (tile placement must not matter)
    and when the weight gradient is run twice.

References are float64 torch on the GPU (the same operations as layer_ref and the autograd chain
of test_bnconv_bwd).  Each case prints its worst |err| / S per pass and mode (pytest -s)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.test_gpu_kernels import L, LAYERS, layer_ref, make_layer_inputs, stream  # noqa: F401

pytestmark = pytest.mark.gpu

MODES = (0, 1, 2, 3, 4, 5, 6)
# elementwise tau per conv precision mode: fp32-level arithmetic (FMA, 3xTF32 and its BF16-corrected
# variants, whose per-product error is <= 2^-18) and plain TF32 (operands rounded to 10 bits)
TAU = {m: (2e-3 if m == 1 else 1e-5) for m in MODES}
# (closest fp32-level case, measured on a B200: convt4's mean-100 input channel, 7.6e-6 in eval mode
# and 9.0e-6 in train mode (bar 1.9e-5 there from the yardstick) in every mode including FMA -- the
# BatchNorm apply x*scale + shift rounds at |x| ~ 100 for a result of order 1; torch in float32 is
# at 6.3e-6 on the same case)
# fp64 reductions of fp32 values the kernel itself wrote (epilogue statistics, border sums),
# relative to the sum of the absolute values of the terms: the in-CTA partials are fp32
RED_TOL = 1e-5
ATOMIC_TOL = 1e-12          # the same fp64 sums in another atomic order
# The same sums when the tiles are spread over the CTAs differently (chunked batch): the FMA forward
# kernels' statistics and every kernel's border sums are fp32 per thread over ALL of a CTA's tiles
# before the fp64 stage, so which tiles share a CTA changes their rounding (measured <= 1.1e-8 on a
# B200).  The tensor-core forward statistics go to fp64 after every tile and hold ATOMIC_TOL.
REGROUP_TOL = 1e-7
GUARD = 64 * 1024           # bytes of guard band on each side of every output
SENTINEL = 0x7FBADBAD       # a NaN as fp32; two of them are a NaN as fp64
TINY = 1e-300


def b_trip(l):
    """Smallest odd B >= 1031 with B * h^2 >= 2 * (8 * 148) * 512, h = the smaller side of the
    layer: at least two trips per CTA for any tile of <= 512 pixels at <= 8 CTAs per SM."""
    name, ci, co, s, h, tr = LAYERS[l]
    ho = h if s == 1 else (2 * h if tr else h // 2)
    hm = min(h, ho)
    B = max(1031, -(-2 * 8 * 148 * 512 // (hm * hm)))
    return B | 1


def h_out(l):
    name, ci, co, s, h, tr = LAYERS[l]
    return h if s == 1 else (2 * h if tr else h // 2)


# ------------------------------------------------------------------------------------- guard bands
class Guarded:
    """`n` elements of `dtype` inside a buffer with GUARD bytes of sentinel on each side."""

    def __init__(self, n, dtype, shape=None):
        esz = torch.empty((), dtype=dtype).element_size()
        assert (n * esz) % 4 == 0
        self.g = GUARD // 4
        self.nw = n * esz // 4
        self.raw = torch.full((2 * self.g + self.nw,), SENTINEL, dtype=torch.int32, device="cuda")
        body = self.raw[self.g:self.g + self.nw]
        self.t = body.view(dtype)
        if shape is not None:
            self.t = self.t.view(shape)

    def ptr(self):
        return self.t.data_ptr()

    def guards_ok(self):
        return bool((self.raw[:self.g] == SENTINEL).all()) and bool((self.raw[self.g + self.nw:] == SENTINEL).all())


def guarded_like(values, dtype=None):
    """A guarded buffer holding a copy of `values` (prefill)."""
    g = Guarded(values.numel(), dtype or values.dtype, tuple(values.shape))
    g.t.copy_(values)
    return g


def bits_equal(a, b):
    """Bitwise equality of two fp32 / fp64 tensors (NaN-safe)."""
    it = torch.int32 if a.element_size() == 4 else torch.int64
    return torch.equal(a.contiguous().view(it), b.contiguous().view(it))


# ------------------------------------------------------------------------------- error measures
def worst_ratio(got, ref, S):
    """max over elements of |got - ref| / S (0 where both the error and S are 0; NaN propagates)."""
    err = (got.double() - ref).abs()
    r = err / S.clamp_min(TINY)
    r = torch.where(err == 0, torch.zeros_like(r), r)
    return float(r.max())


def red_ratio(got, ref, S):
    return worst_ratio(got, ref, S)


class Report:
    """Worst ratios of one case; asserted at the end so that every pass and mode is printed."""

    def __init__(self, tag):
        self.tag = tag
        self.fail = []

    def check(self, what, mode, ratio, bar):
        print("CONF %-34s %-14s mode %d  worst %.3e  bar %.3e" % (self.tag, what, mode, ratio, bar))
        if not ratio <= bar:
            self.fail.append("%s mode %d: worst |err|/S %.3e > bar %.3e" % (what, mode, ratio, bar))

    def require(self, what, mode, ok):
        if not ok:
            self.fail.append("%s mode %d" % (what, mode))

    def done(self):
        assert not self.fail, "%s:\n  %s" % (self.tag, "\n  ".join(self.fail))


def bar_of(mode, yard):
    return max(TAU[mode], 3.0 * yard)


# ------------------------------------------------------------------------------------ references
def conv_op(l, x, w, b=None):
    name, ci, co, s, h, tr = LAYERS[l]
    if tr:
        return F.conv_transpose2d(x, w, b, stride=s, padding=1, output_padding=s - 1)
    return F.conv2d(x, w, b, stride=s, padding=1)


def wgrad_op(l, X, A, wshape):
    """d/dW of <conv(X, W), A>: the weight-gradient operation on given tensors."""
    w0 = torch.zeros(wshape, dtype=X.dtype, device=X.device, requires_grad=True)
    return torch.autograd.grad(conv_op(l, X, w0), w0, A)[0]


def dgrad_op(l, W, A, xshape):
    """d/dX of <conv(X, W), A>: the data-gradient operation."""
    x0 = torch.zeros(xshape, dtype=W.dtype, device=W.device, requires_grad=True)
    return torch.autograd.grad(conv_op(l, x0, W), x0, A)[0]


def border_sums_ref(t, mode):
    """The nine per-channel sums of ava_b200_dz_border_sums, float64 [9, C]."""
    t = t.double()
    if mode == 0:
        parts = [t.sum((0, 2, 3)), t[:, :, 0, :].sum((0, 2)), t[:, :, -1, :].sum((0, 2)),
                 t[:, :, :, 0].sum((0, 2)), t[:, :, :, -1].sum((0, 2)), t[:, :, 0, 0].sum(0),
                 t[:, :, 0, -1].sum(0), t[:, :, -1, 0].sum(0), t[:, :, -1, -1].sum(0)]
    else:
        parts = [t[:, :, 0::2, 0::2].sum((0, 2, 3)), t[:, :, 0::2, 1::2].sum((0, 2, 3)),
                 t[:, :, 1::2, 0::2].sum((0, 2, 3)), t[:, :, 1::2, 1::2].sum((0, 2, 3)),
                 t[:, :, -1, 0::2].sum((0, 2)), t[:, :, -1, 1::2].sum((0, 2)),
                 t[:, :, 0::2, -1].sum((0, 2)), t[:, :, 1::2, -1].sum((0, 2)), t[:, :, -1, -1].sum(0)]
    return torch.stack(parts)


def tsum_mode_of_prev(l):
    return 1 if (l >= 1 and LAYERS[l - 1][5] and LAYERS[l - 1][3] == 2) else 0


def make_case(l, B, family, seed):
    """float64 inputs (fp32-representable) on the GPU: x, dz, w, b, gamma, beta, rm, rv.
    gauss: today's N(0.3, 0.7^2) inputs.  relu / relu_dzscale: per-channel relu(N(mu_c, 1)),
    mu_c in [-0.5, 0.5], channel 1 all zeros, channel 2 mean 100 std 1 (layer 0: U[0, 1] with
    30 % exact zeros); relu_dzscale also scales dz's channels over 2^-20 .. 1."""
    name, ci, co, s, h, tr = LAYERS[l]
    cuda = torch.device("cuda")
    if family == "gauss":
        x, w, b, gamma, beta, rm, rv = make_layer_inputs(l, B, seed)
        x = x.to(cuda)
    else:
        _, w, b, gamma, beta, rm, rv = make_layer_inputs(l, 1, seed)
        g = torch.Generator(device=cuda).manual_seed(seed)
        if ci == 1:
            x = torch.rand(B, 1, h, h, generator=g, device=cuda, dtype=torch.float64)
            x[torch.rand(x.shape, generator=g, device=cuda, dtype=torch.float64) < 0.3] = 0.0
        else:
            mu = torch.rand(ci, generator=g, device=cuda, dtype=torch.float64) - 0.5
            x = torch.relu(torch.randn(B, ci, h, h, generator=g, device=cuda, dtype=torch.float64)
                           + mu.view(1, ci, 1, 1))
            x[:, 1] = 0.0
            x[:, 2] = 100.0 + torch.randn(B, h, h, generator=g, device=cuda, dtype=torch.float64)
        x = x.float().double()
    ho = h_out(l)
    gd = torch.Generator(device=cuda).manual_seed(seed + 1)
    dz = torch.randn(B, co, ho, ho, generator=gd, device=cuda, dtype=torch.float64) + 0.1
    if family == "relu_dzscale" and co > 1:
        dz = dz * torch.pow(2.0, -20.0 * torch.arange(co, device=cuda, dtype=torch.float64) / (co - 1)).view(1, co, 1, 1)
    dz = dz.float().double()
    w, b, gamma, beta = (t.to(cuda) for t in (w, b, gamma, beta))
    # eval-mode buffers near the batch's own statistics (a model's running averages)
    bm = x.mean((0, 2, 3))
    bv = x.var((0, 2, 3), unbiased=False)
    gr = torch.Generator(device=cuda).manual_seed(seed + 2)
    rm = (bm + 0.1 * bv.sqrt() * torch.randn(ci, generator=gr, device=cuda, dtype=torch.float64)).float().double()
    rv = (bv * (0.5 + torch.rand(ci, generator=gr, device=cuda, dtype=torch.float64)) + 1e-3).float().double()
    return x, dz, w, b, gamma, beta, rm, rv


def stats_block(x):
    ci = x.shape[1]
    st = torch.zeros(64, dtype=torch.float64, device="cuda")
    st[:ci] = x.sum((0, 2, 3))
    st[32:32 + ci] = (x * x).sum((0, 2, 3))
    return st


def prefill(n, salt):
    """Known non-zero values for ACCUMULATED outputs."""
    return 0.25 * (torch.arange(n, dtype=torch.float64, device="cuda") % 13 + 1) * (1 + salt)


class NoTF32:
    """The float32 yardstick runs without TF32 (cudnn.allow_tf32 defaults to True)."""

    def __enter__(self):
        self.saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False

    def __exit__(self, *a):
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = self.saved


@pytest.fixture
def no_tf32():
    with NoTF32():
        yield


def forward_refs(l, x, w, b, gamma, beta, rm, rv, train):
    """float64 reference, its absolute-value bound S and the float32 yardstick's worst ratio."""
    xn, y = layer_ref(l, x, w, b, gamma, beta, train, rm, rv)
    S = conv_op(l, xn.abs(), w.abs(), b.abs())
    f = [t.float() for t in (x, w, b, gamma, beta, rm, rv)]
    _, y32 = layer_ref(l, *f[:5], train, f[5], f[6])
    return y, S, worst_ratio(y32, y, S)


def backward_refs(l, x, dz, w, b, gamma, beta):
    """float64 autograd of bn(x) -> conv for the upstream gradient dz, with the bounds S."""
    name, ci, co, s, h, tr = LAYERS[l]
    N = x.shape[0] * h * h
    out = {}
    for dt in (torch.float64, torch.float32):
        xx, ww, bb = (t.to(dt).requires_grad_(True) for t in (x, w, b))
        xn = F.batch_norm(xx, None, None, gamma.to(dt), beta.to(dt), training=True, eps=1e-5)
        z = conv_op(l, xn, ww, bb)
        gx, gw, gb, g = torch.autograd.grad(z, (xx, ww, bb, xn), dz.to(dt))
        mean = x.mean((0, 2, 3), keepdim=True)
        r = dict(dx=gx.double(), dw=gw.double(), db=gb.double(),
                 dbeta=g.double().sum((0, 2, 3)), dgc=(g * (xx.detach() - mean.to(dt))).sum((0, 2, 3)).double())
        out[dt] = r
    ref = out[torch.float64]
    mean = x.mean((0, 2, 3))
    var = x.var((0, 2, 3), unbiased=False)
    invstd = 1.0 / torch.sqrt(var + 1e-5)
    xc = (x - mean.view(1, ci, 1, 1)).abs()
    gabs = dgrad_op(l, w.abs(), dz.abs(), x.shape)
    p = gamma * invstd
    c1 = ref["dbeta"] / N
    q = -gamma * invstd ** 3 * ref["dgc"] / N
    v = lambda t: t.view(1, ci, 1, 1)      # noqa: E731
    S = dict(dx=v(p.abs()) * (gabs + v(c1.abs())) + v(q.abs()) * xc,
             dbeta=gabs.sum((0, 2, 3)), dgc=(gabs * xc).sum((0, 2, 3)),
             db=dz.abs().sum((0, 2, 3)))
    # dw = gamma*invstd * sum dz*(x-mean)_pad + beta * T: the same two terms on absolute values
    wdim = (0 if tr else 1)
    shp = [1, 1, 1, 1]
    shp[wdim] = ci
    S["dw"] = ((gamma * invstd).abs().view(shp) * wgrad_op(l, xc, dz.abs(), w.shape)
               + beta.abs().view(shp) * wgrad_op(l, torch.ones_like(x), dz.abs(), w.shape))
    ref["S"] = S
    ref["dx_masked"] = ref["dx"] * (x > 0)
    y32 = out[torch.float32]
    ref["yard"] = {k: worst_ratio(y32[k], ref[k], S[k]) for k in ("dw", "db", "dbeta", "dgc")}
    ref["yard"]["dx"] = worst_ratio(y32["dx"] * (x > 0), ref["dx_masked"], S["dx"])
    ref["yard"]["dx nomask"] = worst_ratio(y32["dx"], ref["dx"], S["dx"])
    return ref


# ------------------------------------------------------------------------------ the kernel calls
def run_fwd(Lb, l, B, x32, w32, b32, g32, be32, stats_in, rm32, rv32, train, ho, with_stats=True, stats_pre=None):
    name, ci, co, s, h, tr = LAYERS[l]
    y = Guarded(B * co * ho * ho, torch.float32, (B, co, ho, ho))
    st = guarded_like(stats_pre) if with_stats else None
    Lb.call("ava_b200_bnconv_fwd", l, B, x32.data_ptr(), y.ptr(), w32.data_ptr(), b32.data_ptr(),
            g32.data_ptr(), be32.data_ptr(), stats_in.data_ptr(), rm32.data_ptr(), rv32.data_ptr(),
            1 if train else 0, st.ptr() if st is not None else None, stream())
    return y, st


def run_wgrad(Lb, l, B, dz32, x32, w32, g32, be32, stats_in, tsums, dstats_pre):
    name, ci, co, s, h, tr = LAYERS[l]
    wshape = (ci, co, 3, 3) if tr else (co, ci, 3, 3)
    gw = Guarded(int(np.prod(wshape)), torch.float32, wshape)
    gw.t.fill_(float("nan"))                      # OVERWRITTEN
    gb = Guarded(co, torch.float32)
    gb.t.fill_(float("nan"))
    dst = guarded_like(dstats_pre)                # ACCUMULATED
    ws = Guarded(int(Lb.lib().ava_b200_bnconv_bwd_weight_ws(l, B)) // 4, torch.float32)
    Lb.call("ava_b200_bnconv_bwd_weight", l, B, dz32.data_ptr(), x32.data_ptr(), w32.data_ptr(), g32.data_ptr(),
            be32.data_ptr(), stats_in.data_ptr(), tsums.data_ptr(), gw.ptr(), gb.ptr(), dst.ptr(), ws.ptr(),
            stream())
    return gw, gb, dst, ws


def run_bwd_data(Lb, l, B, dz32, w32, x32, g32, stats_in, dstats, mask, tsums_pre):
    name, ci, co, s, h, tr = LAYERS[l]
    out = Guarded(B * ci * h * h, torch.float32, (B, ci, h, h))
    ts = guarded_like(tsums_pre) if tsums_pre is not None else None
    Lb.call("ava_b200_bnconv_bwd_data", l, B, dz32.data_ptr(), w32.data_ptr(), x32.data_ptr(), g32.data_ptr(),
            stats_in.data_ptr(), dstats.data_ptr(), mask, out.ptr(), ts.ptr() if ts is not None else None,
            stream())
    return out, ts


def set_mode(Lb, mode):
    Lb.call("ava_b200_set_conv_precision", mode)


# ------------------------------------------------------------------------------------ conformance
BATCHES = ("1", "64", "1024", "trip")
FAMILIES = ("gauss", "relu", "relu_dzscale")


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("bsel", BATCHES)
@pytest.mark.parametrize("l", range(14))
def test_layer_conformance(L, no_tf32, l, bsel, family):
    """Forward (train; eval at B <= 1024), weight gradient and data gradient of one layer in all
    seven conv precision modes against float64, elementwise, with guard bands and the header's
    ACCUMULATED / OVERWRITTEN contracts.  At B_trip the batch is also run as two unequal chunks."""
    name, ci, co, s, h, tr = LAYERS[l]
    B = b_trip(l) if bsel == "trip" else int(bsel)
    seed = 1000 + 37 * l + 7 * FAMILIES.index(family)
    x, dz, w, b, gamma, beta, rm, rv = make_case(l, B, family, seed)
    ho = h_out(l)
    rep = Report("%s B=%d %s" % (name, B, family))
    x32, dz32, w32, b32, g32, be32, rm32, rv32 = (t.float().contiguous() for t in (x, dz, w, b, gamma, beta, rm, rv))
    stats_in = stats_block(x)
    do_fwd = family != "relu_dzscale"     # (that family differs from relu in dz only)

    fwd = {}
    if do_fwd:
        fwd[True] = forward_refs(l, x, w, b, gamma, beta, rm, rv, True)
        if bsel != "trip":
            fwd[False] = forward_refs(l, x, w, b, gamma, beta, rm, rv, False)
    bw = backward_refs(l, x, dz, w, b, gamma, beta)
    tmode = 1 if (tr and s == 2) else 0
    tsums_dz = torch.zeros(9, 32, dtype=torch.float64, device="cuda")
    tsums_dz[:, :co] = border_sums_ref(dz, tmode)
    tsums_dz = tsums_dz.reshape(288)
    # the layer's BatchNorm-backward reductions as the weight-gradient pass delivers them
    dstats_ref = torch.zeros(64, dtype=torch.float64, device="cuda")
    dstats_ref[:ci] = bw["dbeta"]
    dstats_ref[32:32 + ci] = bw["dgc"]
    pmode = tsum_mode_of_prev(l)
    st_pre, ds_pre, ts_pre = prefill(64, 0), prefill(64, 1), prefill(288, 2)
    chan = torch.arange(64, device="cuda") % 32
    mask_zero = (x == 0)

    try:
        for mode in MODES:
            set_mode(L, mode)
            # ---------------- forward
            for train in (True, False):
                if train not in fwd:
                    continue
                y_ref, S, yard = fwd[train]
                y, st = run_fwd(L, l, B, x32, w32, b32, g32, be32, stats_in, rm32, rv32, train, ho,
                                stats_pre=st_pre)
                y0, _ = run_fwd(L, l, B, x32, w32, b32, g32, be32, stats_in, rm32, rv32, train, ho,
                                with_stats=False)
                torch.cuda.synchronize()
                what = "fwd" if train else "fwd_eval"
                rep.check(what, mode, worst_ratio(y.t, y_ref, S), bar_of(mode, yard))
                rep.require(what + " guard bands", mode, y.guards_ok() and st.guards_ok() and y0.guards_ok())
                rep.require(what + " stats_out=NULL changes y", mode, bits_equal(y.t, y0.t))
                # stats_out: ACCUMULATED onto the prefill; slots [co, 32) and [32 + co, 64) untouched
                own = (chan < co)
                rep.require(what + " stats_out slots beyond co written", mode,
                            bits_equal(st.t[~own], st_pre[~own]))
                yd = y.t.double()
                sums = torch.cat([yd.sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))])
                abss = torch.cat([yd.abs().sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))])
                rep.check(what + " stats_out", mode,
                          red_ratio(st.t[own] - st_pre[own], sums, abss), RED_TOL)
                if bsel == "trip" and mode in (0, 1, 6):
                    # two unequal chunks (count ratio not a power of two: coefficients round
                    # differently, so the elementwise bound applies), statistics into one block
                    b1 = (B - 1) // 2
                    yc = Guarded(B * co * ho * ho, torch.float32, (B, co, ho, ho))
                    stc = guarded_like(st_pre)
                    keep = []           # (the scaled statistics must outlive the asynchronous calls)
                    for lo, hi in ((0, b1), (b1, B)):
                        n = hi - lo
                        keep.append(stats_in * (n / B))
                        L.call("ava_b200_bnconv_fwd", l, n, x32[lo:hi].data_ptr(), yc.t[lo:hi].data_ptr(),
                               w32.data_ptr(), b32.data_ptr(), g32.data_ptr(), be32.data_ptr(),
                               keep[-1].data_ptr(), rm32.data_ptr(), rv32.data_ptr(),
                               1 if train else 0, stc.ptr(), stream())
                    torch.cuda.synchronize()
                    rep.check(what + " 2 chunks", mode, worst_ratio(yc.t, y_ref, S), bar_of(mode, yard))
                    rep.require(what + " 2 chunks guard bands", mode, yc.guards_ok() and stc.guards_ok())
                    ycd = yc.t.double()
                    sums_c = torch.cat([ycd.sum((0, 2, 3)), (ycd * ycd).sum((0, 2, 3))])
                    rep.check(what + " 2 chunks stats", mode,
                              red_ratio(stc.t[own] - st_pre[own], sums_c, abss), RED_TOL)
                    del yc, stc, ycd
                del y, y0, st, yd
            # ---------------- weight gradient
            gw, gb, dst, ws = run_wgrad(L, l, B, dz32, x32, w32, g32, be32, stats_in, tsums_dz, ds_pre)
            torch.cuda.synchronize()
            yard = bw["yard"]
            rep.check("dw", mode, worst_ratio(gw.t, bw["dw"], bw["S"]["dw"]), bar_of(mode, yard["dw"]))
            rep.check("db", mode, worst_ratio(gb.t, bw["db"], bw["S"]["db"]), bar_of(mode, yard["db"]))
            rep.check("dstats sum g", mode, worst_ratio(dst.t[:ci] - ds_pre[:ci], bw["dbeta"], bw["S"]["dbeta"]),
                      bar_of(mode, yard["dbeta"]))
            rep.check("dstats sum g(x-m)", mode,
                      worst_ratio(dst.t[32:32 + ci] - ds_pre[32:32 + ci], bw["dgc"], bw["S"]["dgc"]),
                      bar_of(mode, yard["dgc"]))
            rep.require("wgrad guard bands (dw, db, dstats, workspace)", mode,
                        gw.guards_ok() and gb.guards_ok() and dst.guards_ok() and ws.guards_ok())
            own_i = chan < ci
            rep.require("dstats slots beyond ci written", mode, bits_equal(dst.t[~own_i], ds_pre[~own_i]))
            if B >= 64:
                # run to run: static tile assignment and a fixed-order second stage
                gw2, gb2, dst2, _ = run_wgrad(L, l, B, dz32, x32, w32, g32, be32, stats_in, tsums_dz, ds_pre)
                torch.cuda.synchronize()
                rep.require("dw / db bit-identical run to run", mode,
                            bits_equal(gw.t, gw2.t) and bits_equal(gb.t, gb2.t))
                dabs = torch.cat([bw["S"]["dbeta"] + ds_pre[:ci], bw["S"]["dgc"] + ds_pre[32:32 + ci]])
                rep.check("dstats run to run", mode,
                          red_ratio(torch.cat([dst2.t[:ci], dst2.t[32:32 + ci]]),
                                    torch.cat([dst.t[:ci], dst.t[32:32 + ci]]).double(), dabs), ATOMIC_TOL)
                del gw2, gb2, dst2
            del gw, gb, dst, ws
            # ---------------- data gradient (BatchNorm backward + the previous layer's ReLU mask)
            for mask in (1, 0):
                out, ts = run_bwd_data(L, l, B, dz32, w32, x32, g32, stats_in, dstats_ref, mask,
                                       ts_pre if (mask and l >= 1) else None)
                torch.cuda.synchronize()
                ref = bw["dx_masked"] if mask else bw["dx"]
                what = "dx" if mask else "dx nomask"
                rep.check(what, mode, worst_ratio(out.t, ref, bw["S"]["dx"]), bar_of(mode, bw["yard"][what]))
                rep.require(what + " guard bands", mode, out.guards_ok() and (ts is None or ts.guards_ok()))
                if mask:
                    # [x > 0]: exactly +0.0 wherever the previous layer's output is 0
                    rep.require("dx not exactly 0 where x == 0", mode,
                                bool((out.t.view(torch.int32)[mask_zero] == 0).all()))
                if ts is not None:
                    tref = border_sums_ref(out.t, pmode)
                    tabs = border_sums_ref(out.t.abs(), pmode)
                    t2 = ts.t.view(9, 32)
                    p2 = ts_pre.view(9, 32)
                    rep.check("dx border sums", mode, red_ratio(t2[:, :ci] - p2[:, :ci], tref, tabs), RED_TOL)
                    rep.require("border sums beyond ci written", mode, bits_equal(t2[:, ci:], p2[:, ci:]))
                if bsel == "trip" and mode in (0, 1, 6) and mask:
                    b1 = (B - 1) // 2
                    oc = Guarded(B * ci * h * h, torch.float32, (B, ci, h, h))
                    keep = []
                    for lo, hi in ((0, b1), (b1, B)):
                        n = hi - lo
                        keep += [stats_in * (n / B), dstats_ref * (n / B)]
                        L.call("ava_b200_bnconv_bwd_data", l, n, dz32[lo:hi].data_ptr(), w32.data_ptr(),
                               x32[lo:hi].data_ptr(), g32.data_ptr(), keep[-2].data_ptr(), keep[-1].data_ptr(),
                               1, oc.t[lo:hi].data_ptr(), None, stream())
                    torch.cuda.synchronize()
                    rep.check("dx 2 chunks", mode, worst_ratio(oc.t, ref, bw["S"]["dx"]),
                              bar_of(mode, bw["yard"]["dx"]))
                    rep.require("dx 2 chunks guard bands", mode, oc.guards_ok())
                    del oc
                del out, ts
    finally:
        set_mode(L, 0)
    rep.done()


# ------------------------------------------------------------------------- chunk invariance
@pytest.mark.parametrize("l", range(14))
def test_chunk_invariance(L, l):
    """B = 1024 in one call and as 16 calls of 64 images with stats_in / dstats scaled by 1/16:
    the BatchNorm coefficients are then bitwise identical (both scalings are powers of two), so
    every element must come out bit for bit the same whichever CTA and trip computed it; the
    fp64 statistics and border sums agree to REGROUP_TOL (ATOMIC_TOL where only the atomic order
    can differ) of their absolute sums."""
    name, ci, co, s, h, tr = LAYERS[l]
    B, NC = 1024, 16
    bc = B // NC
    x, dz, w, b, gamma, beta, rm, rv = make_case(l, B, "relu", 5000 + l)
    ho = h_out(l)
    x32, dz32, w32, b32, g32, be32, rm32, rv32 = (t.float().contiguous() for t in (x, dz, w, b, gamma, beta, rm, rv))
    stats_in = stats_block(x)
    gd = torch.Generator(device="cuda").manual_seed(77 + l)
    dstats = torch.zeros(64, dtype=torch.float64, device="cuda")
    dstats[:ci] = torch.randn(ci, generator=gd, device="cuda", dtype=torch.float64) * 0.1 * B * h * h
    dstats[32:32 + ci] = torch.randn(ci, generator=gd, device="cuda", dtype=torch.float64) * 0.1 * B * h * h
    pmode = tsum_mode_of_prev(l)
    rep = Report("%s chunks 16x64" % name)
    try:
        for mode in MODES:
            set_mode(L, mode)
            for train in (True, False):
                yf = torch.empty(B, co, ho, ho, device="cuda")
                yc = torch.empty_like(yf)
                sf = prefill(64, 0)
                sc = prefill(64, 0)
                L.call("ava_b200_bnconv_fwd", l, B, x32.data_ptr(), yf.data_ptr(), w32.data_ptr(), b32.data_ptr(),
                       g32.data_ptr(), be32.data_ptr(), stats_in.data_ptr(), rm32.data_ptr(), rv32.data_ptr(),
                       1 if train else 0, sf.data_ptr(), stream())
                s16 = stats_in / NC
                for k in range(NC):
                    L.call("ava_b200_bnconv_fwd", l, bc, x32[k * bc:].data_ptr(), yc[k * bc:].data_ptr(),
                           w32.data_ptr(), b32.data_ptr(), g32.data_ptr(), be32.data_ptr(), s16.data_ptr(),
                           rm32.data_ptr(), rv32.data_ptr(), 1 if train else 0, sc.data_ptr(), stream())
                torch.cuda.synchronize()
                what = "fwd" if train else "fwd_eval"
                rep.require(what + " y not bit-identical", mode, bits_equal(yf, yc))
                yd = yf.double()
                own = torch.cat([torch.arange(co), 32 + torch.arange(co)]).cuda()
                abss = torch.cat([yd.abs().sum((0, 2, 3)), (yd * yd).sum((0, 2, 3))]) + prefill(64, 0)[own]
                tc_stats = mode != 0 and 1 <= l <= 12
                rep.check(what + " stats_out", mode, red_ratio(sc[own], sf[own], abss),
                          ATOMIC_TOL if tc_stats else REGROUP_TOL)
            of = torch.empty(B, ci, h, h, device="cuda")
            oc = torch.empty_like(of)
            tf = prefill(288, 2)
            tc = prefill(288, 2)
            tp = lambda t: t.data_ptr() if l >= 1 else None     # noqa: E731
            L.call("ava_b200_bnconv_bwd_data", l, B, dz32.data_ptr(), w32.data_ptr(), x32.data_ptr(), g32.data_ptr(),
                   stats_in.data_ptr(), dstats.data_ptr(), 1, of.data_ptr(), tp(tf), stream())
            s16, d16 = stats_in / NC, dstats / NC
            for k in range(NC):
                L.call("ava_b200_bnconv_bwd_data", l, bc, dz32[k * bc:].data_ptr(), w32.data_ptr(),
                       x32[k * bc:].data_ptr(), g32.data_ptr(), s16.data_ptr(), d16.data_ptr(), 1,
                       oc[k * bc:].data_ptr(), tp(tc), stream())
            torch.cuda.synchronize()
            rep.require("dx not bit-identical", mode, bits_equal(of, oc))
            if l >= 1:
                tabs = border_sums_ref(of.abs(), pmode) + prefill(288, 2).view(9, 32)[:, :ci]
                rep.check("dx border sums", mode,
                          red_ratio(tc.view(9, 32)[:, :ci], tf.view(9, 32)[:, :ci].double(), tabs), REGROUP_TOL)
    finally:
        set_mode(L, 0)
    rep.done()


# ------------------------------------------------------------------------- bn_relu_bwd_apply
@pytest.mark.parametrize("B", [1, 64, 1024])
def test_bn_relu_bwd_apply_seam(L, B):
    """The fc1 -> conv7 seam form the model uses: C = 32, HW = 256, W = 16, no BatchNorm, ReLU
    mask of conv7's output, `out` aliasing `g`, border sums of the result accumulated on the way.
    Without BatchNorm the result is g itself where a > 0 and exactly +0.0 elsewhere."""
    C, H, W = 32, 16, 16
    gen = torch.Generator(device="cuda").manual_seed(B)
    a = torch.relu(torch.randn(B, C, H, W, generator=gen, device="cuda")
                   + (torch.rand(C, generator=gen, device="cuda") - 0.5).view(1, C, 1, 1))
    a[:, 3] = 0.0
    g = torch.randn(B, C, H, W, generator=gen, device="cuda") + 0.1
    buf = Guarded(g.numel(), torch.float32, g.shape)
    buf.t.copy_(g)
    ts_pre = prefill(288, 3)
    ts = guarded_like(ts_pre)
    L.call("ava_b200_bn_relu_bwd_apply", buf.ptr(), a.data_ptr(), None, None, None, B, C, H * W, 1, buf.ptr(),
           ts.ptr(), W, stream())
    ts_k = torch.zeros(288, dtype=torch.float64, device="cuda")
    L.call("ava_b200_dz_border_sums", buf.ptr(), B, C, H, W, 0, ts_k.data_ptr(), stream())
    torch.cuda.synchronize()
    assert buf.guards_ok() and ts.guards_ok()
    assert bits_equal(buf.t, torch.where(a > 0, g, torch.zeros_like(g)))
    got = (ts.t - ts_pre).view(9, 32)
    tabs = border_sums_ref(buf.t.abs(), 0)
    assert red_ratio(got, border_sums_ref(buf.t, 0), tabs) <= RED_TOL
    assert red_ratio(got, ts_k.view(9, 32), tabs) <= RED_TOL


@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("B", [1, 64, 1024])
@pytest.mark.parametrize("C,H", [(32, 16), (24, 32), (8, 64)])
def test_bn_relu_bwd_apply_batchnorm(L, B, C, H, relu):
    """The BatchNorm form: out = [a > 0] * (p*(g - c1) + q*(a - mean)) against float64, elementwise
    relative to |p|(|g| + |c1|) + |q||a - mean|; ReLU-like `a` with an all-zero channel and a
    channel of mean 100; masked entries exactly +0.0."""
    W = H
    gen = torch.Generator(device="cuda").manual_seed(B * 10 + C + relu)
    a = torch.relu(torch.randn(B, C, H, W, generator=gen, device="cuda", dtype=torch.float64)
                   + (torch.rand(C, generator=gen, device="cuda", dtype=torch.float64) - 0.5).view(1, C, 1, 1))
    a[:, 1] = 0.0
    a[:, 2] = 100.0 + torch.randn(B, H, W, generator=gen, device="cuda", dtype=torch.float64)
    a = a.float().double()
    g = (torch.randn(B, C, H, W, generator=gen, device="cuda", dtype=torch.float64) + 0.1).float().double()
    gamma = (torch.rand(C, generator=gen, device="cuda", dtype=torch.float64) + 0.5).float().double()
    N = B * H * W
    stats = stats_block(a)
    mean = a.mean((0, 2, 3))
    var = a.var((0, 2, 3), unbiased=False)
    dstats = torch.zeros(64, dtype=torch.float64, device="cuda")
    dstats[:C] = g.sum((0, 2, 3))
    dstats[32:32 + C] = (g * (a - mean.view(1, C, 1, 1))).sum((0, 2, 3))
    invstd = 1.0 / torch.sqrt(var + 1e-5)
    p = gamma * invstd
    c1 = dstats[:C] / N
    q = -gamma * invstd ** 3 * dstats[32:32 + C] / N
    v = lambda t: t.view(1, C, 1, 1)      # noqa: E731
    ref = v(p) * (g - v(c1)) + v(q) * (a - v(mean))
    S = v(p.abs()) * (g.abs() + v(c1.abs())) + v(q.abs()) * (a - v(mean)).abs()
    if relu:
        ref = ref * (a > 0)
    a32, g32, gm32 = a.float(), g.float(), gamma.float()
    out = Guarded(g.numel(), torch.float32, g.shape)
    ts_pre = prefill(288, 4)
    ts = guarded_like(ts_pre)
    L.call("ava_b200_bn_relu_bwd_apply", g32.data_ptr(), a32.data_ptr(), gm32.data_ptr(), stats.data_ptr(),
           dstats.data_ptr(), B, C, H * W, relu, out.ptr(), ts.ptr(), W, stream())
    torch.cuda.synchronize()
    assert out.guards_ok() and ts.guards_ok()
    # fp64 coefficient math, one rounding to fp32 at the end
    r = worst_ratio(out.t, ref, S)
    print("CONF bn_relu_bwd_apply B=%d C=%d HW=%d relu=%d  worst %.3e" % (B, C, H * W, relu, r))
    assert r <= 1e-6
    if relu:
        assert bool((out.t.view(torch.int32)[a == 0] == 0).all())
    got = (ts.t - ts_pre).view(9, 32)
    assert red_ratio(got[:, :C], border_sums_ref(out.t, 0), border_sums_ref(out.t.abs(), 0)) <= RED_TOL
    assert bits_equal(ts.t.view(9, 32)[:, C:], ts_pre.view(9, 32)[:, C:])
