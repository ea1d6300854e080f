"""Conformance of the dense (Linear) layers -- csrc/gemm.cu (SIMT GEMM, split-K, bias gradients) and
csrc/gemm_tc.cu (tcgen05) -- as the training step calls them.

Compared with the dense tests of tests/test_gpu_kernels.py (max-norm errors, made-up shapes, M <= 130
on the SIMT path and M = 128 / 256 on the tcgen05 path) these tests
  * take every call from STEP TABLE, a restatement of the dense calls in models/vae.py (shapes,
    leading dimensions, group strides, activation, precision, mask / db present), and check by
    recording one train_step that the model still makes exactly those calls;
  * run each call at batches that reach every path: the SIMT kernel with split-K from 37-way to none
    (FMA or, at precision 1, mma.sync TF32), and the tcgen05 kernel with 16-, 4-, 2-way split-K and
    the direct epilogue; Z = 32 and Z = 7 (odd leading dimensions: scalar loads, no vector stores);
  * bound every output ELEMENT: |got - ref64| <= bar * S, S = the same product on absolute values,
    bar = max(tau(precision), 3 x the worst ratio of float32 torch without TF32);
  * feed ReLU-like inputs (half exact zeros, an all-zero column, a column of mean 100), upstream
    gradients whose columns span 2^-20 .. 1, and masks holding +0.0, -0.0 and negative values;
  * put every output and the workspace inside NaN guard bands, and check the header's contracts:
    only owned elements change, dw / db overwrite, the masked form is a select (bit-identical to the
    unmasked form on a pre-masked dY, and to a dY holding NaN where the mask is off), every call is
    bit-identical run to run, a short workspace is an error on the tcgen05 path and one split on the
    SIMT path, accumulate = 1 is rejected.

References are float64 torch on the GPU.  With pytest -s each case prints one line per pass and
precision: CONF <layer.pass B Z inputs> <what and path: kernel and split-K count> mode <precision>
worst <max |err|/S> bar <bar>.  The path is computed by this file's restatement of pick_splits /
tc_splits / mma_terms (gemm.cu, gemm_tc.cu), so that what a case covers can be read off the output."""
import ctypes
import importlib
import math

import pytest
import torch

from tests.test_gpu_conv_conformance import SENTINEL, Guarded, NoTF32, Report, bits_equal, worst_ratio
from tests.test_gpu_kernels import PKG, L, stream  # noqa: F401

pytestmark = pytest.mark.gpu

FWD, BWD_W, BWD_D = "ava_b200_linear_fwd", "ava_b200_linear_bwd_weight", "ava_b200_linear_bwd_data"
BIAS = "ava_b200_bias_grads"
# argument names in ABI order (include/ava_b200.h)
ARGS = {
    FWD: ("x", "ldx", "w", "b", "y", "ldy", "M", "N", "K", "act", "groups", "x_gs", "w_gs", "b_gs", "y_gs",
          "precision", "ws", "ws_bytes", "stream"),
    BWD_W: ("dy", "lddy", "ymask", "x", "ldx", "dw", "db", "M", "N", "K", "groups", "dy_gs", "x_gs", "dw_gs",
            "db_gs", "precision", "ws", "ws_bytes", "stream"),
    BWD_D: ("dy", "lddy", "ymask", "w", "dx", "lddx", "M", "N", "K", "groups", "dy_gs", "w_gs", "dx_gs",
            "accumulate", "precision", "ws", "ws_bytes", "stream"),
}
POINTERS = {"x", "w", "b", "y", "dy", "ymask", "dw", "db", "dx", "ws"}
NOT_COMPARED = {"ws_bytes", "stream"}    # the scratch size is checked against the call's need instead

# elementwise tau per precision: fp32 FMA and 3xTF32 at fp32 level; single TF32.  At precision 1 the
# SIMT kernel's mma.sync reads the fp32 bit patterns as TF32 (the low 13 bits are dropped, not
# rounded), so one product can be off by up to 2^-9 = 1.95e-3 of its size: a one-row contraction
# (bwd_weight at batch 1) sits right there.  The tcgen05 pre-pass rounds (cvt.rna): half of that.
TAU = {0: 1e-5, 1: 2e-3, 2: 1e-5}
EXP_ULPS = 4 * 2.0 ** -24               # expf: <= 2 ulp
TC_LAYERS = ("fc1", "fc2", "fc7", "fc8")
NSM = 148                                # kNumSMs (common.cuh)


# ------------------------------------------------------------------------------------ step table
def _fwd(layer, M, N, K, ldx, ldy, act, prec, groups=1, x_gs=0, w_gs=0, b_gs=0, y_gs=0, x_off=0):
    """One ava_b200_linear_fwd call; x_off: element offset of x from the start of its buffer."""
    return dict(fn=FWD, layer=layer, ldx=ldx, ldy=ldy, M=M, N=N, K=K, act=act, groups=groups, x_gs=x_gs,
                w_gs=w_gs, b_gs=b_gs, y_gs=y_gs, precision=prec, x_off=x_off)


def _bwd(layer, M, N, K, lddy, ldx, lddx, masked, prec, groups=1, dy_gs=0, x_gs=0, w_gs=0, b_gs=0, dx_gs=0):
    """VAE._linear_bwd with a bias job list: bwd_weight with db = NULL, then bwd_data."""
    return [dict(fn=BWD_W, layer=layer, lddy=lddy, ymask=masked, ldx=ldx, db=False, M=M, N=N, K=K,
                 groups=groups, dy_gs=dy_gs, x_gs=x_gs, dw_gs=w_gs, db_gs=b_gs, precision=prec),
            dict(fn=BWD_D, layer=layer, lddy=lddy, ymask=masked, lddx=lddx, M=M, N=N, K=K, groups=groups,
                 dy_gs=dy_gs, w_gs=w_gs, dx_gs=dx_gs, accumulate=0, precision=prec)]


def encoder_fwd(B, Z, tc):
    """VAE._encode_native: fc1, fc2, fc31|32|33 as one [192, 256] layer, fc41|42|43 as a strided
    batch of three [Z, 64] layers on the three 64-wide slices of h3 into the heads buffer [B, 3Z]."""
    return [_fwd("fc1", B, 1024, 8192, 8192, 1024, 1, tc),
            _fwd("fc2", B, 256, 1024, 1024, 256, 1, tc),
            _fwd("fc31", B, 192, 256, 256, 192, 1, 0),
            _fwd("fc41|42|43", B, Z, 64, 192, 3 * Z, 0, 0, groups=3, x_gs=64, w_gs=Z * 64, b_gs=Z, y_gs=Z)]


def decoder_fwd(B, Z, tc):
    """VAE._decode_native: fc5 .. fc8."""
    return [_fwd("fc5", B, 64, Z, Z, 64, 1, 0),
            _fwd("fc6", B, 256, 64, 64, 256, 1, 0),
            _fwd("fc7", B, 1024, 256, 256, 1024, 1, tc),
            _fwd("fc8", B, 8192, 1024, 1024, 8192, 1, tc)]


def encode_fc43(B, Z):
    """VAE.encode: d = exp(fc43(h3[:, 128:])), input 128 floats (512 bytes) into h3, output ld Z."""
    return _fwd("fc43", B, Z, 64, 192, Z, 2, 0, x_off=128)


def bwd_decoder(B, Z, tc):
    """VAE._bwd_decoder: fc8 .. fc5 (fc8's output gradient comes unmasked from convt1's backward)."""
    return (_bwd("fc8", B, 8192, 1024, 8192, 1024, 1024, False, tc)
            + _bwd("fc7", B, 1024, 256, 1024, 256, 256, True, tc)
            + _bwd("fc6", B, 256, 64, 256, 64, 64, True, 0)
            + _bwd("fc5", B, 64, Z, 64, Z, Z, True, 0))


def bwd_dense_encoder(B, Z, tc):
    """VAE._bwd_dense_encoder: the heads (unmasked, grouped), fc31, fc2, fc1."""
    return (_bwd("fc41|42|43", B, Z, 64, 3 * Z, 192, 192, False, 0, groups=3, dy_gs=Z, x_gs=64, w_gs=Z * 64,
                 b_gs=Z, dx_gs=64)
            + _bwd("fc31", B, 192, 256, 192, 256, 256, True, 0)
            + _bwd("fc2", B, 256, 1024, 256, 1024, 1024, True, tc)
            + _bwd("fc1", B, 1024, 8192, 1024, 8192, 8192, True, tc))


def bias_jobs_decoder(B, Z):
    """The decoder segment's ava_b200_bias_grads jobs: (name, masked, ld, M, N)."""
    return [("fc8", False, 8192, B, 8192), ("fc7", True, 1024, B, 1024), ("fc6", True, 256, B, 256),
            ("fc5", True, 64, B, 64)]


def bias_jobs_encoder(B, Z):
    """The dense encoder segment's jobs; the grouped heads layer is one job of N = 3Z columns."""
    return [("fc41|42|43", False, 3 * Z, B, 3 * Z), ("fc31", True, 192, B, 192), ("fc2", True, 256, B, 256),
            ("fc1", True, 1024, B, 1024)]


def step_table(B, Z, tc):
    """Every dense call of one train step, in issue order."""
    return (encoder_fwd(B, Z, tc) + decoder_fwd(B, Z, tc) + bwd_decoder(B, Z, tc)
            + [dict(fn=BIAS, jobs=bias_jobs_decoder(B, Z))] + bwd_dense_encoder(B, Z, tc)
            + [dict(fn=BIAS, jobs=bias_jobs_encoder(B, Z))])


def signature(c):
    """What the step table says about a call: integer arguments, and NULL or not for pointers."""
    if c["fn"] == BIAS:
        return (BIAS, tuple(("ptr", "ptr" if m else "NULL", "ptr", ld, M, N) for _, m, ld, M, N in c["jobs"]))
    return (c["fn"],) + tuple((a, ("ptr" if c.get(a, True) else "NULL") if a in POINTERS else c[a])
                              for a in ARGS[c["fn"]] if a not in NOT_COMPARED)


class _Job(ctypes.Structure):
    """ava_b200_bias_job (include/ava_b200.h)."""
    _fields_ = [("dy", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("db", ctypes.c_void_p),
                ("ld", ctypes.c_int), ("M", ctypes.c_int), ("N", ctypes.c_int)]


class Recorder:
    """_lib.PROFILER hook: keeps the arguments of every dense call as it is issued."""

    def __init__(self):
        self.calls = []

    def begin(self, name, args):
        if name in ARGS:
            self.calls.append((name, tuple(args)))
        elif name == BIAS:
            arr, n = args[0], args[1]
            jobs = [(j.dy, j.mask, j.db, j.ld, j.M, j.N) for j in arr[:n]]
            self.calls.append((name, (jobs,) + tuple(args[1:])))

    def end(self, name, args):
        pass


def recorded_signature(name, args):
    if name == BIAS:
        return (BIAS, tuple(tuple("ptr" if v else "NULL" for v in j[:3]) + tuple(j[3:]) for j in args[0]))
    return (name,) + tuple((a, ("ptr" if v else "NULL") if a in POINTERS else int(v))
                           for a, v in zip(ARGS[name], args) if a not in NOT_COMPARED)


def _arg(name, args, a):
    return args[ARGS[name].index(a)]


@pytest.mark.parametrize("B", (64, 128))
def test_step_dense_calls_match_table(L, B):
    """One eager train_step and one encode() of the model, recorded through _lib.PROFILER: the dense
    calls, in order, are exactly those of the step table (every integer argument, NULL-ness of every
    pointer), and every scratch buffer the step passes is large enough for the call."""
    vae_mod = importlib.import_module(PKG + ".models.vae")
    torch.manual_seed(B)
    model = vae_mod.VAE(save_dir="", device_name="cuda", cuda_graphs=False)
    Z, tc = model.z_dim, model._tc
    x = torch.rand(B, 128, 128, device="cuda")
    rec, rec_enc = Recorder(), Recorder()
    try:
        L.PROFILER = rec
        model.train_step(x)
        L.PROFILER = rec_enc
        model.encode(x)
    finally:
        L.PROFILER = None
    torch.cuda.synchronize()
    lib = L.lib()
    for got_calls, want_calls in ((rec.calls, step_table(B, Z, tc)),
                                  (rec_enc.calls, encoder_fwd(B, Z, tc) + [encode_fc43(B, Z)])):
        got = [recorded_signature(n, a) for n, a in got_calls]
        want = [signature(c) for c in want_calls]
        for i, (g, w) in enumerate(zip(got, want)):
            assert g == w, "dense call %d differs from the step table:\n  model %s\n  table %s" % (i, g, w)
        assert len(got) == len(want), "model made %d dense calls, the table lists %d" % (len(got), len(want))
        for name, args in got_calls:
            if name == BIAS:
                jobs, n, ws, ws_bytes = args[0], args[1], args[2], args[3]
                arr = (_Job * n)(*[_Job(*j) for j in jobs])
                assert ws and ws_bytes >= lib.ava_b200_bias_grads_ws_bytes(arr, n)
            else:
                M, N, K = (_arg(name, args, a) for a in ("M", "N", "K"))
                assert _arg(name, args, "ws") and _arg(name, args, "ws_bytes") >= lib.ava_b200_linear_ws_bytes(M, N, K)
    # encode(): fc43 reads h3 (fc31's output) 512 bytes in
    fc31 = [a for n, a in rec_enc.calls if n == FWD][2]
    fc43 = [a for n, a in rec_enc.calls if n == FWD][4]
    assert _arg(FWD, fc43, "x") - _arg(FWD, fc31, "y") == 512


# ------------------------------------------------------------------ which path a call takes
def simt_splits(M, N, K, groups, ws_bytes):
    """pick_splits + run_gemm (gemm.cu) for the GEMM C[M, N] = A[M, K] B[K, N]."""
    tiles = -(-M // 64) * -(-N // 64) * groups
    s = 1
    if tiles < 2 * NSM:
        s = min(max(1, 4 * NSM // tiles), max(1, K // 128), 64)
    if s > 1 and (ws_bytes is None or ws_bytes < s * groups * M * N * 4):
        s = 1
    kc = -(-(-(-K // s)) // 16) * 16
    return -(-K // kc)


def tc_supported(M, N, K):
    return M > 0 and N > 0 and K > 0 and M % 128 == 0 and N % 128 == 0 and K % 32 == 0


def tc_splits(M, N, K):
    tiles, kb, s = (M // 128) * (N // 128), K // 32, 1
    while tiles * s < NSM and s * 2 <= kb // 8 and s < 16:
        s *= 2
    return s


def tc_ws_bytes(M, N, K):
    """Workspace of the tcgen05 GEMM: TF32 hi/lo copies of both operands + split-K partials."""
    return (2 * M * K + 2 * N * K + tc_splits(M, N, K) * M * N) * 4 + 4096


def colsum_splits(M, N, ws_bytes):
    cb, s = -(-N // 32), 1
    while cb * s < 2 * NSM and M // (s * 2) >= 64:
        s *= 2
    return 1 if (ws_bytes is None or ws_bytes < s * N * 4) else s


def gemm_dims(c):
    M, N, K = c["M"], c["N"], c["K"]
    return {FWD: (M, N, K), BWD_D: (M, K, N), BWD_W: (N, K, M)}[c["fn"]]


def path_of(c, prec, ws_bytes):
    """(kernel, split-K count) of a call at a precision and workspace size."""
    gm = gemm_dims(c)
    if prec >= 1 and c["groups"] == 1 and tc_supported(*gm):
        return "tcgen05", tc_splits(*gm)
    mma = prec == 1 and c["groups"] == 1 and c["N"] * c["K"] >= (1 << 18)
    return ("simt-mma" if mma else "simt-fma"), simt_splits(*gm, c["groups"], ws_bytes)


# ------------------------------------------------------------------------------------- inputs
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _f64(*shape, gen, rand=torch.randn):
    return rand(*shape, generator=gen, device="cuda", dtype=torch.float64)


def make_x(G, M, K, family, gen):
    """Layer input [G, M, K]: N(0, 0.5^2), or ReLU-like: relu(N(mu_k, 1)), mu_k in [-0.5, 0.5] (half
    exact zeros), column 1 all zero, column 2 of mean 100."""
    if family == "gauss":
        x = 0.5 * _f64(G, M, K, gen=gen)
    else:
        x = torch.relu(_f64(G, M, K, gen=gen) + (_f64(G, 1, K, gen=gen, rand=torch.rand) - 0.5))
        x[:, :, 1] = 0.0
        x[:, :, 2] = 100.0 + _f64(G, M, gen=gen)
    return x.float().double()


def make_dy(G, M, N, family, gen):
    """Upstream gradient [G, M, N]: N(0.1, 1); ReLU-like family: columns scaled over 2^-20 .. 1."""
    dy = _f64(G, M, N, gen=gen) + 0.1
    if family != "gauss" and N > 1:
        dy = dy * torch.pow(2.0, -20.0 * torch.arange(N, device="cuda", dtype=torch.float64) / (N - 1))
    return dy.float().double()


def make_mask(G, M, N, gen):
    """A ReLU mask source [G, M, N]: positive values, +0.0, -0.0 and negative values."""
    u = _f64(G, M, N, gen=gen, rand=torch.rand)
    v = _f64(G, M, N, gen=gen, rand=torch.rand) + 0.25
    z = torch.zeros_like(v)
    m = torch.where(u < 0.5, v, torch.where(u < 0.65, z, torch.where(u < 0.8, -z, -v)))
    m.view(-1)[:3] = torch.tensor([0.0, -0.0, -1.0], dtype=torch.float64, device="cuda")
    return m.float().double()


def view3(flat, off, ld, gs, G, M, C):
    """The [G, M, C] operand at element offset `off` of `flat`, rows `ld` apart, groups `gs` apart."""
    return flat.as_strided((G, M, C), (gs, ld, 1), flat.storage_offset() + off)


def buffer_with(logical, off, ld, gs, n, gen):
    """A float64 buffer of n elements, Gaussian junk around `logical` placed at (off, ld, gs)."""
    buf = _f64(n, gen=gen).float().double()
    view3(buf, off, ld, gs, *logical.shape).copy_(logical)
    return buf


def owned(n, off, ld, gs, G, M, C):
    own = torch.zeros(n, dtype=torch.bool, device="cuda")
    view3(own, off, ld, gs, G, M, C).fill_(True)
    return own


def untouched(g, own):
    """Every element of the guarded buffer outside `own` still holds the sentinel, and the guard bands."""
    return g.guards_ok() and bool((g.t.reshape(-1).view(torch.int32)[~own] == SENTINEL).all())


def bar_of(prec, yard):
    return max(TAU[prec], 3.0 * yard)


def workspace(L, c, ws_null):
    if ws_null:
        return None, None, 0
    nb = int(L.lib().ava_b200_linear_ws_bytes(c["M"], c["N"], c["K"]))
    assert nb % 4 == 0
    ws = Guarded(nb // 4, torch.float32)
    return ws, ws.ptr(), nb


def ws_ok(ws):
    return ws is None or ws.guards_ok()


# ------------------------------------------------------------------------------------- runners
def run_fwd_case(L, rep, c, precs, family, seed, ws_null=False):
    G, M, N, K = c["groups"], c["M"], c["N"], c["K"]
    ldx, ldy, x_gs, y_gs, off = c["ldx"], c["ldy"], c["x_gs"], c["y_gs"], c["x_off"]
    gen = _gen(seed)
    x = make_x(G, M, K, family, gen)
    w = (_f64(G, N, K, gen=gen) / math.sqrt(K)).float().double()
    b = (0.1 * _f64(G, N, gen=gen)).float().double()
    xbuf = buffer_with(x, off, ldx, x_gs, off + M * ldx, gen)
    wbuf = buffer_with(w, 0, K, c["w_gs"], (G - 1) * c["w_gs"] + N * K, gen)
    bbuf = buffer_with(b.view(G, 1, N), 0, N, c["b_gs"], (G - 1) * c["b_gs"] + N, gen)
    pre = x @ w.transpose(1, 2) + b[:, None, :]
    S = x.abs() @ w.abs().transpose(1, 2) + b.abs()[:, None, :]
    with NoTF32():
        pre32 = x.float() @ w.float().transpose(1, 2) + b.float()[:, None, :]
    yard = worst_ratio(pre32, pre, S)
    x32, w32, b32 = xbuf.float(), wbuf.float(), bbuf.float()
    ny = M * ldy
    own = owned(ny, 0, ldy, y_gs, G, M, N)
    for prec in precs:
        ws, wsp, wsb = workspace(L, c, ws_null)
        ys = []
        for _ in range(2):
            y = Guarded(ny, torch.float32)
            L.call(FWD, x32.data_ptr() + 4 * off, ldx, w32.data_ptr(), b32.data_ptr(), y.ptr(), ldy, M, N, K,
                   c["act"], G, x_gs, c["w_gs"], c["b_gs"], y_gs, prec, wsp, wsb, stream())
            ys.append(y)
        torch.cuda.synchronize()
        got = view3(ys[0].t, 0, ldy, y_gs, G, M, N)
        kern, sp = path_of(c, prec, None if ws_null else wsb)
        bar = bar_of(prec, yard)
        if c["act"] == 2:
            # |got - exp(ref)| <= exp(ref) * (bar * S + 4 * 2^-24)
            e = torch.exp(pre)
            r = ((got.double() - e).abs() - e * EXP_ULPS).clamp_min(0) / (e * S).clamp_min(1e-300)
            ratio = float(r.max())
        else:
            ratio = worst_ratio(got, torch.relu(pre) if c["act"] == 1 else pre, S)
        rep.check("y %s x%d" % (kern, sp), prec, ratio, bar)
        rep.require("y: guard bands, or elements outside y written", prec,
                    untouched(ys[0], own) and untouched(ys[1], own) and ws_ok(ws))
        rep.require("y not bit-identical run to run", prec, bits_equal(ys[0].t, ys[1].t))


def run_bwd_case(L, rep, cw, cd, precs, family, seed, ws_null=False):
    """bwd_weight as the step runs it (db = NULL), again with db, and bwd_data; with a mask also on a
    pre-masked dY without mask and on a dY holding NaN wherever the mask is off."""
    G, M, N, K = cw["groups"], cw["M"], cw["N"], cw["K"]
    lddy, dy_gs, ldx, x_gs = cw["lddy"], cw["dy_gs"], cw["ldx"], cw["x_gs"]
    lddx, dx_gs, w_gs, db_gs = cd["lddx"], cd["dx_gs"], cd["w_gs"], cw["db_gs"]
    masked = cw["ymask"]
    gen = _gen(seed)
    x = make_x(G, M, K, family, gen)
    w = (_f64(G, N, K, gen=gen) / math.sqrt(K)).float().double()
    dy = make_dy(G, M, N, family, gen)
    ndy = M * lddy
    dybuf = buffer_with(dy, 0, lddy, dy_gs, ndy, gen)
    xbuf = buffer_with(x, 0, ldx, x_gs, M * ldx, gen)
    wbuf = buffer_with(w, 0, K, w_gs, (G - 1) * w_gs + N * K, gen)
    if masked:
        mask = make_mask(G, M, N, gen)
        mbuf = buffer_with(mask, 0, lddy, dy_gs, ndy, gen)
        on = mask > 0
        dym = torch.where(on, dy, torch.zeros_like(dy))
        pre_buf = dybuf.clone()
        view3(pre_buf, 0, lddy, dy_gs, G, M, N).copy_(dym)
        nan_buf = dybuf.clone()
        view3(nan_buf, 0, lddy, dy_gs, G, M, N).copy_(torch.where(on, dy, torch.full_like(dy, float("nan"))))
        pre32, nan32, m32 = pre_buf.float(), nan_buf.float(), mbuf.float()
    else:
        dym = dy
    ref = dict(dx=dym @ w, dw=dym.transpose(1, 2) @ x, db=dym.sum(1))
    S = dict(dx=dym.abs() @ w.abs(), dw=dym.abs().transpose(1, 2) @ x.abs(), db=dym.abs().sum(1))
    with NoTF32():
        d32, w32_, x32_ = dym.float(), w.float(), x.float()
        got32 = dict(dx=d32 @ w32_, dw=d32.transpose(1, 2) @ x32_, db=d32.sum(1))
    yard = {k: worst_ratio(got32[k], ref[k], S[k]) for k in ref}
    dy32, x32, w32 = dybuf.float(), xbuf.float(), wbuf.float()
    nw, nb, nx = (G - 1) * cw["dw_gs"] + N * K, (G - 1) * db_gs + N, M * lddx
    own_w = owned(nw, 0, K, cw["dw_gs"], G, N, K)
    own_b = owned(nb, 0, N, db_gs, G, 1, N)
    own_x = owned(nx, 0, lddx, dx_gs, G, M, K)
    # (dY, mask) pairs: as the step; pre-masked without mask; NaN where the mask is off
    variants = [(dy32, m32 if masked else None)]
    if masked:
        variants += [(pre32, None), (nan32, m32)]
    for prec in precs:
        ws, wsp, wsb = workspace(L, cw, ws_null)
        # ---- weight gradient
        runs = []
        for i, (d, m) in enumerate([variants[0]] + variants):
            gw = Guarded(nw, torch.float32)
            gb = Guarded(nb, torch.float32) if i > 0 else None
            L.call(BWD_W, d.data_ptr(), lddy, m.data_ptr() if m is not None else None, x32.data_ptr(), ldx,
                   gw.ptr(), gb.ptr() if gb is not None else None, M, N, K, G, dy_gs, x_gs, cw["dw_gs"], db_gs,
                   prec, wsp, wsb, stream())
            runs.append((gw, gb))
        torch.cuda.synchronize()
        kern, sp = path_of(cw, prec, None if ws_null else wsb)
        gw, gb = runs[1]
        rep.check("dw %s x%d" % (kern, sp), prec, worst_ratio(view3(gw.t, 0, K, cw["dw_gs"], G, N, K), ref["dw"],
                                                            S["dw"]), bar_of(prec, yard["dw"]))
        rep.check("db colsum x%d" % colsum_splits(M, N, None if ws_null else wsb), prec,
                  worst_ratio(view3(gb.t, 0, N, db_gs, G, 1, N).reshape(G, N), ref["db"], S["db"]),
                  bar_of(prec, yard["db"]))
        rep.require("dw / db: guard bands, or elements outside dw / db written", prec,
                    all(untouched(a, own_w) and (b_ is None or untouched(b_, own_b)) for a, b_ in runs) and ws_ok(ws))
        rep.require("dw differs with db = NULL", prec, bits_equal(runs[0][0].t, gw.t))
        if masked:
            rep.require("dw / db on a pre-masked dY without mask not bit-identical", prec,
                        bits_equal(runs[2][0].t, gw.t) and bits_equal(runs[2][1].t, gb.t))
            rep.require("dw / db with NaN in dY where the mask is off not bit-identical", prec,
                        bits_equal(runs[3][0].t, gw.t) and bits_equal(runs[3][1].t, gb.t))
        del runs, gw, gb
        # ---- data gradient
        outs = []
        for d, m in [variants[0]] + variants:
            dx = Guarded(nx, torch.float32)
            L.call(BWD_D, d.data_ptr(), lddy, m.data_ptr() if m is not None else None, w32.data_ptr(), dx.ptr(),
                   lddx, M, N, K, G, dy_gs, w_gs, dx_gs, 0, prec, wsp, wsb, stream())
            outs.append(dx)
        torch.cuda.synchronize()
        kern, sp = path_of(cd, prec, None if ws_null else wsb)
        rep.check("dx %s x%d" % (kern, sp), prec, worst_ratio(view3(outs[0].t, 0, lddx, dx_gs, G, M, K), ref["dx"],
                                                            S["dx"]), bar_of(prec, yard["dx"]))
        rep.require("dx: guard bands, or elements outside dx written", prec,
                    all(untouched(o, own_x) for o in outs) and ws_ok(ws))
        rep.require("dx not bit-identical run to run", prec, bits_equal(outs[0].t, outs[1].t))
        if masked:
            rep.require("dx on a pre-masked dY without mask not bit-identical", prec, bits_equal(outs[2].t, outs[0].t))
            rep.require("dx with NaN in dY where the mask is off not bit-identical", prec,
                        bits_equal(outs[3].t, outs[0].t))
        del outs


# ------------------------------------------------------------------------------------- cases
B_SIMT = (1, 7, 64, 100, 1000)
B_TC = (128, 1024, 2048, 4096)
B_BIG = 4160          # precision 2, fc1 / fc8 shapes only: SIMT without split-K at the largest shapes
ZS = (32, 7)
FAMILIES = ("gauss", "relu")


def conformance_calls(B, Z):
    """The step table's dense calls, the bwd_weight / bwd_data pair of a layer as one case."""
    tbl = encoder_fwd(B, Z, 2) + decoder_fwd(B, Z, 2) + [encode_fc43(B, Z)]
    out = [(c["layer"], "fwd", (c,)) for c in tbl]
    bw = bwd_decoder(B, Z, 2) + bwd_dense_encoder(B, Z, 2)
    out += [(bw[i]["layer"], "bwd", (bw[i], bw[i + 1])) for i in range(0, len(bw), 2)]
    return out


def _cases():
    """(id, layer, pass, B, Z or None, precisions): every table entry at every B, for Z = 32 and 7;
    an entry whose arguments do not depend on Z runs once (Z = None)."""
    cases = []
    for B in B_SIMT + B_TC + (B_BIG,):
        per_z = {Z: conformance_calls(B, Z) for Z in ZS}
        for i, (layer, kind, _) in enumerate(per_z[ZS[0]]):
            if B == B_BIG and layer not in ("fc1", "fc8"):
                continue
            sigs = {signature(c) for Z in ZS for c in per_z[Z][i][2]}
            zs = ZS if len(sigs) > len(per_z[ZS[0]][i][2]) else (None,)
            precs = (2,) if B == B_BIG else ((0, 1, 2) if layer in TC_LAYERS else (0,))
            for Z in zs:
                cid = "%s.%s-B%d%s" % (layer, kind, B, "" if Z is None else "-Z%d" % Z)
                cases.append(pytest.param(layer, kind, B, Z, precs, id=cid))
    return cases


def run_case(L, layer, kind, B, Z, precs, calls, ws_null=False):
    """Both input families; every family and precision is printed before the first failure is raised."""
    seed = 7919 * B + 31 * (Z or 0) + sum(map(ord, layer + kind))
    reports = []
    for fi, family in enumerate(FAMILIES):
        rep = Report("%s.%s B=%d Z=%s %s" % (layer, kind, B, "32/7" if Z is None else Z, family))
        if kind == "fwd":
            run_fwd_case(L, rep, calls[0], precs, family, seed + fi, ws_null)
        else:
            run_bwd_case(L, rep, calls[0], calls[1], precs, family, seed + fi, ws_null)
        reports.append(rep)
    for rep in reports:
        rep.done()


@pytest.mark.parametrize("layer,kind,B,Z,precs", _cases())
def test_dense_conformance(L, layer, kind, B, Z, precs):
    """One step-table entry at one batch: forward (y), or weight gradient (dw, db) and data gradient
    (dx), elementwise against float64, with guard bands, bitwise run-to-run and mask contracts."""
    calls = {(c[0], c[1]): c[2] for c in conformance_calls(B, 32 if Z is None else Z)}[(layer, kind)]
    run_case(L, layer, kind, B, Z, precs, calls)


@pytest.mark.parametrize("kind", ("fwd", "bwd"))
def test_simt_without_workspace(L, kind):
    """ws = NULL on the SIMT path: one split instead of 37 (fc1 forward at batch 64) or 4 (its data
    gradient), and still within the bound; the forward also at precision 1 (mma.sync TF32; the weight
    gradient would take the tcgen05 path there, which needs its workspace)."""
    calls = {(c[0], c[1]): c[2] for c in conformance_calls(64, 32)}[("fc1", kind)]
    precs = (0, 1) if kind == "fwd" else (0,)
    assert all(path_of(c, p, None)[0] != "tcgen05" for c in calls for p in precs)
    assert max(path_of(c, 0, int(L.lib().ava_b200_linear_ws_bytes(64, 1024, 8192)))[1] for c in calls) > 1
    run_case(L, "fc1", kind, 64, None, precs, calls, ws_null=True)


@pytest.mark.parametrize("B", (7, 100))
def test_grouped_gaps(L, B):
    """A strided batch whose group blocks do not tile the row (ld > groups * block, gaps between the
    blocks of y / dx / db, odd strides): the gaps stay bitwise unchanged and the values meet the bound."""
    Z = 7
    fwd = _fwd("gapped", B, Z, 64, 203, 3 * (Z + 3) + 5, 0, 0, groups=3, x_gs=67, w_gs=Z * 64 + 5, b_gs=Z + 2,
               y_gs=Z + 3)
    run_case(L, "gapped", "fwd", B, Z, (0,), (fwd,))
    bw = _bwd("gapped", B, Z, 64, 3 * (Z + 3) + 5, 203, 203, True, 0, groups=3, dy_gs=Z + 3, x_gs=67,
              w_gs=Z * 64 + 5, b_gs=Z + 2, dx_gs=67)
    run_case(L, "gapped", "bwd", B, Z, (0,), tuple(bw))


# ------------------------------------------------------------------------------------ contracts
def _operands(M, N, K, seed):
    gen = _gen(seed)
    t = lambda *s: _f64(*s, gen=gen).float()       # noqa: E731
    return t(M, K), t(N, K) / math.sqrt(K), t(N), t(M, N)


def test_tc_workspace_one_byte_short(L):
    """A tcgen05-eligible call given one byte less than the tcgen05 GEMM's workspace fails with a
    message and writes nothing (output, db or workspace); with exactly that many bytes it runs."""
    lib = L.lib()
    for fn, (M, N, K), prec in ((FWD, (128, 1024, 8192), 2), (BWD_D, (1024, 8192, 1024), 1),
                                (BWD_W, (128, 1024, 8192), 2)):
        x, w, b, dy = _operands(M, N, K, M + N + K)
        c = dict(fn=fn, M=M, N=N, K=K, groups=1)
        gm = gemm_dims(c)
        assert tc_supported(*gm) and path_of(c, prec, None)[0] == "tcgen05"
        need = tc_ws_bytes(*gm)
        assert need <= lib.ava_b200_linear_ws_bytes(M, N, K)
        for nbytes in (need - 1, need):
            ws = Guarded(need // 4, torch.float32)
            out = Guarded({FWD: M * N, BWD_D: M * K, BWD_W: N * K}[fn], torch.float32)
            db = Guarded(N, torch.float32)
            # an earlier, different error: the message must be this call's
            assert lib.ava_b200_linear_bwd_data(dy.data_ptr(), N, None, w.data_ptr(), out.ptr(), K, M, N, K, 1, 0,
                                                0, 0, 1, 0, None, 0, stream()) != 0
            if fn == FWD:
                rc = lib.ava_b200_linear_fwd(x.data_ptr(), K, w.data_ptr(), b.data_ptr(), out.ptr(), N, M, N, K, 1, 1,
                                             0, 0, 0, 0, prec, ws.ptr(), nbytes, stream())
            elif fn == BWD_D:
                rc = lib.ava_b200_linear_bwd_data(dy.data_ptr(), N, dy.data_ptr(), w.data_ptr(), out.ptr(), K, M, N,
                                                  K, 1, 0, 0, 0, 0, prec, ws.ptr(), nbytes, stream())
            else:
                rc = lib.ava_b200_linear_bwd_weight(dy.data_ptr(), N, dy.data_ptr(), x.data_ptr(), K, out.ptr(),
                                                    db.ptr(), M, N, K, 1, 0, 0, 0, 0, prec, ws.ptr(), nbytes,
                                                    stream())
            torch.cuda.synchronize()
            if nbytes == need:
                assert rc == 0, L.last_error()
                assert not bool(out.t.isnan().any()), "%s with exactly the tcgen05 workspace" % fn
                continue
            msg = L.last_error()
            assert rc != 0 and "workspace" in msg, (fn, rc, msg)
            for g in (ws, out, db):
                nothing = torch.zeros(g.t.numel(), dtype=torch.bool, device="cuda")
                assert untouched(g, nothing), "%s wrote with a short workspace" % fn


def test_bwd_data_rejects_accumulate(L):
    """accumulate = 1 is not supported: ava_b200_linear_bwd_data returns an error and leaves dx alone."""
    M, N, K = 64, 1024, 256
    _, w, _, dy = _operands(M, N, K, 5)
    dx = Guarded(M * K, torch.float32)
    dx.t.copy_(torch.arange(M * K, device="cuda", dtype=torch.float32))
    before = dx.t.clone()
    ws_bytes = int(L.lib().ava_b200_linear_ws_bytes(M, N, K))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    for prec in (0, 2):
        rc = L.lib().ava_b200_linear_bwd_data(dy.data_ptr(), N, None, w.data_ptr(), dx.ptr(), K, M, N, K, 1, 0, 0, 0,
                                              1, prec, ws.data_ptr(), ws_bytes, stream())
        torch.cuda.synchronize()
        assert rc != 0 and "accumulate" in L.last_error()
        assert bits_equal(dx.t, before) and dx.guards_ok()


# ---------------------------------------------------------------------------------- bias grads
BIAS_ROWS = (1, 7, 31, 64, 100, 1000, 1024, 1057, 4160)


@pytest.mark.parametrize("Z", ZS)
@pytest.mark.parametrize("B", BIAS_ROWS)
def test_bias_grads_step_jobs(L, B, Z):
    """ava_b200_bias_grads with the step's two job lists against per-layer float64 column sums of the
    masked gradient (rows below 32 and not a multiple of 32 reach the remainder loop), overwriting a
    NaN prefill, bitwise run to run, and the mask a select (pre-masked dY, NaN dY: bit-identical)."""
    lib = L.lib()
    for segment, jobs in (("decoder", bias_jobs_decoder(B, Z)), ("encoder", bias_jobs_encoder(B, Z))):
        rep = Report("bias_grads %s B=%d Z=%d" % (segment, B, Z))
        gen = _gen(1000 * B + Z + len(segment))
        data = []
        for name, masked, ld, M, N in jobs:
            dy = make_dy(1, M, N, "relu", gen)
            dybuf = buffer_with(dy, 0, ld, 0, M * ld, gen)
            if masked:
                mask = make_mask(1, M, N, gen)
                mbuf = buffer_with(mask, 0, ld, 0, M * ld, gen)
                on = mask > 0
                dym = torch.where(on, dy, torch.zeros_like(dy))
                pre_buf, nan_buf = dybuf.clone(), dybuf.clone()
                view3(pre_buf, 0, ld, 0, 1, M, N).copy_(dym)
                view3(nan_buf, 0, ld, 0, 1, M, N).copy_(torch.where(on, dy, torch.full_like(dy, float("nan"))))
                bufs = (dybuf.float(), mbuf.float(), pre_buf.float(), nan_buf.float())
            else:
                dym = dy
                bufs = (dybuf.float(), None, dybuf.float(), dybuf.float())
            with NoTF32():
                yard = worst_ratio(dym.float().sum(1)[0], dym.sum(1)[0], dym.abs().sum(1)[0])
            data.append((name, ld, M, N, bufs, dym.sum(1)[0], dym.abs().sum(1)[0], yard))

        def run(variant):
            """variant 0: (dY, mask); 1: pre-masked dY, no mask; 2: NaN dY, mask."""
            arr = (_Job * len(jobs))()
            outs = []
            for a, (name, ld, M, N, bufs, _, _, _) in zip(arr, data):
                dyv, mk = bufs[(0, 2, 3)[variant]], (None if variant == 1 else bufs[1])
                db = Guarded(N, torch.float32)
                outs.append(db)
                a.dy, a.mask, a.db = dyv.data_ptr(), (mk.data_ptr() if mk is not None else None), db.ptr()
                a.ld, a.M, a.N = ld, M, N
            need = int(lib.ava_b200_bias_grads_ws_bytes(arr, len(jobs)))
            ws = Guarded(need // 4, torch.float32)
            L.call(BIAS, arr, len(jobs), ws.ptr(), need, stream())
            torch.cuda.synchronize()
            return outs, ws

        first, ws = run(0)
        again, ws2 = run(0)
        premasked, ws3 = run(1)
        nan, ws4 = run(2)
        rep.require("guard bands", 0, all(g.guards_ok() for g in first + again + premasked + nan + [ws, ws2, ws3, ws4]))
        for j, (name, ld, M, N, bufs, ref, S, yard) in enumerate(data):
            sp = 1
            while -(-N // 32) * sp < 8 * NSM and M // (sp * 2) >= 32 and sp < 64:
                sp *= 2
            rep.check("%s x%d" % (name, sp), 0, worst_ratio(first[j].t, ref, S), bar_of(0, yard))
            rep.require("%s not bit-identical run to run" % name, 0, bits_equal(first[j].t, again[j].t))
            rep.require("%s pre-masked without mask not bit-identical" % name, 0, bits_equal(first[j].t, premasked[j].t))
            rep.require("%s NaN where the mask is off not bit-identical" % name, 0, bits_equal(first[j].t, nan[j].t))
        rep.done()
