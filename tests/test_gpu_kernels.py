"""GPU parity tests of the individual kernels, called through the C ABI (ctypes) and
checked against float64 torch CPU references of the same arithmetic."""
import ctypes
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests.helpers import rel_err

pytestmark = pytest.mark.gpu

PKG = "autoencoded-vocal-analysis_b200"
LAYERS = [("conv1", 1, 8, 1, 128, 0), ("conv2", 8, 8, 2, 128, 0), ("conv3", 8, 16, 1, 64, 0),
          ("conv4", 16, 16, 2, 64, 0), ("conv5", 16, 24, 1, 32, 0), ("conv6", 24, 24, 2, 32, 0),
          ("conv7", 24, 32, 1, 16, 0), ("convt1", 32, 24, 1, 16, 1), ("convt2", 24, 24, 2, 16, 1),
          ("convt3", 24, 16, 1, 32, 1), ("convt4", 16, 16, 2, 32, 1), ("convt5", 16, 8, 1, 64, 1),
          ("convt6", 8, 8, 2, 64, 1), ("convt7", 8, 1, 1, 128, 1)]
TOL = 1e-4   # fp32 kernels vs float64 reference (north_star rtol 1e-4)
# conv inner-product arithmetic (ava_b200_set_conv_precision): fp32 FMA and error-compensated
# 3xTF32 on the tensor cores hold the fp32 bar; plain TF32 has its own stated tolerance
# (mode 3: the 3-term product with its two correction terms as half-rate BF16 instructions)
CONV_MODES = [(0, TOL), (2, TOL), (3, TOL), (4, TOL), (5, TOL), (6, TOL), (1, 5e-3)]


@pytest.fixture(params=CONV_MODES, ids=["fp32", "tf32x3", "tf32x3b", "tf32x3c", "tf32x3d", "tf32x3e", "tf32"])
def conv_mode(request, L):
    mode, tol = request.param
    L.call("ava_b200_set_conv_precision", mode)
    yield mode, tol
    L.call("ava_b200_set_conv_precision", 0)


@pytest.fixture(scope="module")
def L():
    lib = importlib.import_module(PKG + "._lib")
    lib.lib()
    return lib


def dev(t, dtype=torch.float32):
    return t.to(dtype).cuda().contiguous()


def stream():
    return torch.cuda.current_stream().cuda_stream


def layer_ref(l, x, w, b, gamma, beta, train, rm, rv):
    name, ci, co, s, h, tr = LAYERS[l]
    xn = F.batch_norm(x, rm.clone(), rv.clone(), gamma, beta, training=train, momentum=0.1, eps=1e-5)
    if tr:
        y = F.conv_transpose2d(xn, w, b, stride=s, padding=1, output_padding=s - 1)
    else:
        y = F.conv2d(xn, w, b, stride=s, padding=1)
    if l != 13:
        y = F.relu(y)
    return xn, y


def make_layer_inputs(l, B, seed):
    name, ci, co, s, h, tr = LAYERS[l]
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, ci, h, h, generator=g, dtype=torch.float64) * 0.7 + 0.3
    wshape = (ci, co, 3, 3) if tr else (co, ci, 3, 3)
    w = torch.randn(wshape, generator=g, dtype=torch.float64) / np.sqrt(9 * ci)
    b = torch.randn(co, generator=g, dtype=torch.float64) * 0.1
    gamma = torch.rand(ci, generator=g, dtype=torch.float64) + 0.5
    beta = torch.randn(ci, generator=g, dtype=torch.float64) * 0.2
    rm = torch.randn(ci, generator=g, dtype=torch.float64) * 0.1
    rv = torch.rand(ci, generator=g, dtype=torch.float64) + 0.5
    # round everything to fp32-representable values so both sides see identical inputs
    return [t.float().double() for t in (x, w, b, gamma, beta, rm, rv)]


# batch sizes of the per-layer tests: 3 (a handful of tiles), 64 and 130 (several waves of tiles per
# CTA, ragged tile counts, many per-CTA partials in the fp64 statistics / weight-gradient reductions);
# the reduced-precision mode is exercised at the small size only
def _batches(mode):
    return (3,) if mode == 1 else (3, 64, 130)


@pytest.mark.parametrize("l", range(14))
@pytest.mark.parametrize("train", [True, False])
def test_bnconv_fwd(L, l, train, conv_mode):
    mode, tol = conv_mode
    name, ci, co, s, h, tr = LAYERS[l]
    for B in _batches(mode):
        if B != 3 and not train:
            continue
        x, w, b, gamma, beta, rm, rv = make_layer_inputs(l, B, 100 + l)
        _, y_ref = layer_ref(l, x, w, b, gamma, beta, train, rm, rv)
        dx, dw, db, dg, dbeta, drm, drv = [dev(t) for t in (x, w, b, gamma, beta, rm, rv)]
        stats = torch.zeros(2 * 64, dtype=torch.float64, device="cuda")
        L.call("ava_b200_channel_stats", dx.data_ptr(), B, ci, h * h, stats.data_ptr(), stream())
        ho = y_ref.shape[-1]
        y = torch.empty(B, co, ho, ho, device="cuda")
        L.call("ava_b200_bnconv_fwd", l, B, dx.data_ptr(), y.data_ptr(), dw.data_ptr(), db.data_ptr(),
               dg.data_ptr(), dbeta.data_ptr(), stats.data_ptr(), drm.data_ptr(), drv.data_ptr(),
               1 if train else 0, stats.data_ptr() + 8 * 64, stream())
        torch.cuda.synchronize()
        assert rel_err(y.cpu().numpy(), y_ref.numpy()) <= tol, B
        st = stats.cpu().numpy()
        # input statistics kernel
        assert rel_err(st[:ci], x.sum(dim=(0, 2, 3)).numpy()) <= 1e-5
        assert rel_err(st[32:32 + ci], (x * x).sum(dim=(0, 2, 3)).numpy()) <= 1e-5
        # epilogue statistics of the output (the next BN's batch statistics)
        assert rel_err(st[64:64 + co], y_ref.sum(dim=(0, 2, 3)).numpy()) <= tol, B
        assert rel_err(st[96:96 + co], (y_ref * y_ref).sum(dim=(0, 2, 3)).numpy()) <= tol, B


def _trimmed_sums_ref(l, dz, h_in):
    """T[co,3,3]: sum of dz over the pixels whose tap partner lies inside the image = the
    weight gradient of the layer w.r.t. an all-ones single input channel (float64)."""
    name, ci, co, s, h, tr = LAYERS[l]
    ones = torch.ones(dz.shape[0], 1, h_in, h_in, dtype=torch.float64)
    if not tr:
        w0 = torch.zeros(co, 1, 3, 3, dtype=torch.float64, requires_grad=True)
        y = F.conv2d(ones, w0, stride=s, padding=1)
    else:
        w0 = torch.zeros(1, co, 3, 3, dtype=torch.float64, requires_grad=True)
        y = F.conv_transpose2d(ones, w0, stride=s, padding=1, output_padding=s - 1)
    (y * dz).sum().backward()
    return w0.grad.reshape(co, 3, 3)


@pytest.mark.parametrize("l", range(14))
def test_bnconv_bwd(L, l, conv_mode):
    """Backward of one fused layer through the C ABI in its three steps (include/ava_b200.h):
    border sums of dz -> weight / bias gradients + the layer's BatchNorm-backward reductions
    (algebraically, from the same centred raw product) -> data gradient with the BatchNorm
    backward and the previous layer's ReLU mask applied in the epilogue.  Reference: float64
    autograd through bn(x) -> conv for the same dz."""
    mode, tol = conv_mode
    name, ci, co, s, h, tr = LAYERS[l]
    for B in _batches(mode):
        x, w, b, gamma, beta, rm, rv = make_layer_inputs(l, B, 200 + l)
        x.requires_grad_(True)
        w.requires_grad_(True)
        b.requires_grad_(True)
        gen = torch.Generator().manual_seed(300 + l)
        xn = F.batch_norm(x, None, None, gamma, beta, training=True, eps=1e-5)
        xn.retain_grad()
        if tr:
            z = F.conv_transpose2d(xn, w, b, stride=s, padding=1, output_padding=s - 1)
        else:
            z = F.conv2d(xn, w, b, stride=s, padding=1)
        ho = z.shape[-1]
        dz = (torch.randn(z.shape, generator=gen, dtype=torch.float64) + 0.1).float().double()
        z.backward(dz)
        g = xn.grad                                   # gradient w.r.t. the BatchNorm output
        xd = x.detach()
        mean_x = xd.mean(dim=(0, 2, 3), keepdim=True)
        stats = torch.zeros(64, dtype=torch.float64)
        stats[:ci] = xd.sum(dim=(0, 2, 3))
        stats[32:32 + ci] = (xd * xd).sum(dim=(0, 2, 3))
        d = lambda t: dev(t)          # noqa: E731
        dx, dw_, dg, dbeta, ddz = d(xd), d(w.detach()), d(gamma), d(beta), d(dz)
        dstats_in = stats.cuda()
        tsums = torch.zeros(288, dtype=torch.float64, device="cuda")
        tmode = 1 if (tr and s == 2) else 0
        L.call("ava_b200_dz_border_sums", ddz.data_ptr(), B, co, ho, ho, tmode, tsums.data_ptr(), stream())
        ws_bytes = L.lib().ava_b200_bnconv_bwd_weight_ws(l, B)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        gw = torch.full(w.shape, 7.0, device="cuda")
        gb = torch.full((co,), 7.0, device="cuda")
        dst = torch.zeros(64, dtype=torch.float64, device="cuda")
        L.call("ava_b200_bnconv_bwd_weight", l, B, ddz.data_ptr(), dx.data_ptr(), dw_.data_ptr(), dg.data_ptr(),
               dbeta.data_ptr(), dstats_in.data_ptr(), tsums.data_ptr(), gw.data_ptr(), gb.data_ptr(),
               dst.data_ptr(), ws.data_ptr(), stream())
        gin = torch.empty(B, ci, h, h, device="cuda")
        # (the epilogue also accumulates the border sums of what it writes: the previous layer's)
        tprev = torch.zeros(288, dtype=torch.float64, device="cuda")
        L.call("ava_b200_bnconv_bwd_data", l, B, ddz.data_ptr(), dw_.data_ptr(), dx.data_ptr(), dg.data_ptr(),
               dstats_in.data_ptr(), dst.data_ptr(), 1, gin.data_ptr(), tprev.data_ptr() if l >= 1 else None,
               stream())
        gin_nomask = torch.empty(B, ci, h, h, device="cuda")
        L.call("ava_b200_bnconv_bwd_data", l, B, ddz.data_ptr(), dw_.data_ptr(), dx.data_ptr(), dg.data_ptr(),
               dstats_in.data_ptr(), dst.data_ptr(), 0, gin_nomask.data_ptr(), None, stream())
        torch.cuda.synchronize()
        if l >= 1:
            # fused border sums == the stand-alone pass over the same tensor
            pmode = 1 if (LAYERS[l - 1][5] and LAYERS[l - 1][3] == 2) else 0
            tref = torch.zeros(288, dtype=torch.float64, device="cuda")
            L.call("ava_b200_dz_border_sums", gin.data_ptr(), B, ci, h, h, pmode, tref.data_ptr(), stream())
            torch.cuda.synchronize()
            tscale = float(gin.double().abs().sum()) / ci
            assert float((tprev - tref).abs().max()) <= 1e-6 * tscale, ("fused tsums", B, pmode)
        # trimmed sums (float64 accumulation of fp32 values: near exact)
        T = _trimmed_sums_ref(l, dz, h)
        ts = tsums.cpu().reshape(9, 32)
        # (fp32 partial sums of 4 neighbours, then float64)
        if tmode == 0:
            assert rel_err(ts[0, :co].numpy(), dz.sum(dim=(0, 2, 3)).numpy()) <= 1e-7
            assert rel_err(ts[1, :co].numpy(), dz[:, :, 0, :].sum(dim=(0, 2)).numpy()) <= 1e-7
            assert rel_err(ts[4, :co].numpy(), dz[:, :, :, -1].sum(dim=(0, 2)).numpy()) <= 1e-7
            assert rel_err(ts[8, :co].numpy(), dz[:, :, -1, -1].sum(dim=0).numpy()) <= 1e-7
        else:
            assert rel_err(ts[1, :co].numpy(), dz[:, :, 0::2, 1::2].sum(dim=(0, 2, 3)).numpy()) <= 1e-7
        assert rel_err(gw.cpu().numpy(), w.grad.numpy()) <= tol, ("dw", B)
        # a bias in front of a BatchNorm has (nearly) zero gradient in the full network: absolute
        # tolerance scaled by the magnitude of the terms that cancel
        dz_scale = np.abs(dz.numpy()).sum() / co
        assert np.abs(gb.cpu().numpy() - b.grad.numpy()).max() <= 1e-6 * dz_scale, ("db", B)
        # the layer's BatchNorm-backward reductions, obtained algebraically
        dbeta_ref = g.sum(dim=(0, 2, 3)).numpy()
        dgc_ref = (g * (xd - mean_x)).sum(dim=(0, 2, 3)).numpy()
        got = dst.cpu().numpy()
        scale = max(np.abs(g.numpy()).sum() / ci, 1e-30)   # cancellation-aware scale
        stol = 1e-5 if mode != 1 else 1e-3
        assert np.abs(got[:ci] - dbeta_ref).max() <= stol * scale, ("dbeta", B)
        assert np.abs(got[32:32 + ci] - dgc_ref).max() <= stol * scale, ("dgamma", B)
        # data gradient through the BatchNorm backward, with and without the ReLU mask of the
        # producing layer ([x > 0]: x has both signs here)
        assert rel_err(gin_nomask.cpu().numpy(), x.grad.numpy()) <= tol, ("dx", B)
        assert rel_err(gin.cpu().numpy(), (x.grad * (xd > 0)).numpy()) <= tol, ("dx masked", B)
        # consistency of the algebra with the reference's own T (all nine taps)
        Wd = w.detach()
        if not tr:
            sum_g = torch.einsum("oikl,okl->i", Wd, T)
        else:
            sum_g = torch.einsum("iokl,okl->i", Wd, T)
        assert np.abs(sum_g.numpy() - dbeta_ref).max() <= 1e-9 * scale


@pytest.mark.parametrize("M,N,K,act,groups", [(64, 1024, 8192, 1, 1), (7, 256, 1024, 1, 1),
                                             (5, 192, 256, 1, 1), (33, 32, 64, 0, 3),
                                             (130, 8192, 1024, 1, 1), (3, 64, 32, 2, 1),
                                             (9, 20, 64, 0, 3)])
def test_linear_fwd_bwd(L, M, N, K, act, groups):
    gen = torch.Generator().manual_seed(M * 7 + N)
    G = groups
    x = (torch.randn(M, G * K, generator=gen, dtype=torch.float64) * 0.5).float().double()
    w = (torch.randn(G, N, K, generator=gen, dtype=torch.float64) / np.sqrt(K)).float().double()
    b = (torch.randn(G, N, generator=gen, dtype=torch.float64) * 0.1).float().double()
    w.requires_grad_(True)
    b.requires_grad_(True)
    x.requires_grad_(True)
    ys = []
    for g in range(G):
        pre = F.linear(x[:, g * K:(g + 1) * K], w[g], b[g])
        ys.append(F.relu(pre) if act == 1 else (torch.exp(pre) if act == 2 else pre))
    y_ref = torch.cat(ys, dim=1)
    dY = torch.randn(M, G * N, generator=gen, dtype=torch.float64).float().double()
    dx_, dw_, db_ = dev(x.detach()), dev(w.detach()), dev(b.detach())
    y = torch.empty(M, G * N, device="cuda")
    ws_bytes = max(L.lib().ava_b200_linear_ws_bytes(M, N, K), 1 << 20)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    L.call("ava_b200_linear_fwd", dx_.data_ptr(), G * K, dw_.data_ptr(), db_.data_ptr(), y.data_ptr(),
           G * N, M, N, K, act, G, K, N * K, N, N, 0, ws.data_ptr(), ws_bytes, stream())
    torch.cuda.synchronize()
    assert rel_err(y.cpu().numpy(), y_ref.detach().numpy()) <= TOL
    if act == 2:
        return
    # backward: upstream gradient dY w.r.t. the post-activation output
    (y_ref * dY).sum().backward()
    ddy = dev(dY)
    mask = y.data_ptr() if act == 1 else None
    gw = torch.full((G, N, K), 3.0, device="cuda")
    gb = torch.full((G, N), 3.0, device="cuda")
    gx = torch.full((M, G * K), 3.0, device="cuda")
    L.call("ava_b200_linear_bwd_weight", ddy.data_ptr(), G * N, mask, dx_.data_ptr(), G * K,
           gw.data_ptr(), gb.data_ptr(), M, N, K, G, N, K, N * K, N, 0, ws.data_ptr(), ws_bytes,
           stream())
    L.call("ava_b200_linear_bwd_data", ddy.data_ptr(), G * N, mask, dw_.data_ptr(), gx.data_ptr(),
           G * K, M, N, K, G, N, N * K, K, 0, 0, ws.data_ptr(), ws_bytes, stream())
    torch.cuda.synchronize()
    assert rel_err(gw.cpu().numpy(), w.grad.numpy()) <= TOL
    assert rel_err(gb.cpu().numpy(), b.grad.numpy()) <= TOL
    assert rel_err(gx.cpu().numpy(), x.grad.numpy()) <= TOL


@pytest.mark.parametrize("B,Z", [(1, 32), (64, 32), (13, 8), (5, 64)])
def test_latent_and_recon(L, B, Z):
    from oracle import vae_oracle
    gen = torch.Generator().manual_seed(B + Z)
    heads = (torch.randn(B, 3 * Z, generator=gen, dtype=torch.float64) * 0.5).float().double()
    ew = torch.randn(B, 1, generator=gen, dtype=torch.float64).float().double()
    ed = torch.randn(B, Z, generator=gen, dtype=torch.float64).float().double()
    gz = torch.randn(B, Z, generator=gen, dtype=torch.float64).float().double()
    heads.requires_grad_(True)
    mu, u, logd = heads[:, :Z], heads[:, Z:2 * Z], heads[:, 2 * Z:]
    d = torch.exp(logd)
    z = vae_oracle.rsample(mu, u.unsqueeze(-1), d, ew, ed)
    ent = vae_oracle.entropy(u.unsqueeze(-1), d).sum()
    # loss part that depends on the heads: 1/2 sum z^2 - H + <gz, z> (gz = decoder gradient)
    (0.5 * (z * z).sum() - ent + (gz * z).sum()).backward()
    dh, dew, ded, dgz = dev(heads.detach()), dev(ew), dev(ed), dev(gz)
    zz = torch.empty(B, Z, device="cuda")
    dd = torch.empty(B, Z, device="cuda")
    acc = torch.zeros(4, dtype=torch.float64, device="cuda")
    L.call("ava_b200_latent_fwd", dh.data_ptr(), dew.data_ptr(), ded.data_ptr(), B, Z, zz.data_ptr(),
           dd.data_ptr(), acc.data_ptr(), stream())
    gh = torch.empty(B, 3 * Z, device="cuda")
    L.call("ava_b200_latent_bwd", dh.data_ptr(), dew.data_ptr(), ded.data_ptr(), zz.data_ptr(),
           dgz.data_ptr(), B, Z, gh.data_ptr(), stream())
    # recon
    n = B * 16384
    x = torch.rand(n, generator=gen, dtype=torch.float64).float().double()
    xr = (x + torch.randn(n, generator=gen, dtype=torch.float64)).float().double()
    g = torch.empty(n, device="cuda")
    dx_, dxr_ = dev(x), dev(xr)
    ts = torch.zeros(9 * 32, dtype=torch.float64, device="cuda")
    L.call("ava_b200_recon", dx_.data_ptr(), dxr_.data_ptr(), n, 10.0, g.data_ptr(),
           acc.data_ptr(), ts.data_ptr(), 128, 128, stream())
    # the border sums accumulated while g was written == a separate pass over g
    ts_ref = torch.zeros(9 * 32, dtype=torch.float64, device="cuda")
    L.call("ava_b200_dz_border_sums", g.data_ptr(), B, 1, 128, 128, 0, ts_ref.data_ptr(), stream())
    torch.cuda.synchronize()
    scale = float(g.abs().sum())
    assert float((ts - ts_ref).abs().max()) <= 1e-6 * scale
    assert float(ts_ref.abs().max()) > 0
    loss = torch.zeros(1, device="cuda")
    lsum = torch.full((1,), 5.0, dtype=torch.float64, device="cuda")
    L.call("ava_b200_elbo_finalize", acc.data_ptr(), Z, 16384, 10.0, loss.data_ptr(), lsum.data_ptr(),
           stream())
    torch.cuda.synchronize()
    a = acc.cpu().numpy()
    assert rel_err(zz.cpu().numpy(), z.detach().numpy()) <= 1e-6
    assert rel_err(dd.cpu().numpy(), d.detach().numpy()) <= 1e-6
    assert abs(a[0] - (z * z).sum().item()) <= 1e-5 * (z * z).sum().item()
    assert abs(a[2] - ent.item()) <= 1e-5 * abs(ent.item())
    sse = ((x - xr) ** 2).sum().item()
    assert abs(a[1] - sse) <= 1e-5 * sse
    assert rel_err(g.cpu().numpy(), (10.0 * (xr - x)).numpy()) <= 1e-6
    assert rel_err(gh.cpu().numpy(), heads.grad.numpy()) <= 1e-5
    want = 0.5 * ((z * z).sum().item() + Z * np.log(2 * np.pi)) \
        + 0.5 * 16384 * np.log(2 * np.pi / 10.0) + 0.5 * 10.0 * sse - ent.item()
    assert abs(loss.item() - want) <= 1e-6 * abs(want)
    assert abs(lsum.item() - 5.0 - want) <= 1e-6 * abs(want)


@pytest.mark.parametrize("M", [7, 64, 1024])
def test_bias_grads_batched(L, M):
    """ava_b200_bias_grads: the bias gradients of several Linear layers (column sums of the masked
    upstream gradient, incl. a grouped layer's adjacent column blocks as one job) in two launches,
    against float64 sums; bit-identical run to run (fixed-order reduction)."""
    import ctypes

    class Job(ctypes.Structure):
        _fields_ = [("dy", ctypes.c_void_p), ("mask", ctypes.c_void_p), ("db", ctypes.c_void_p),
                    ("ld", ctypes.c_int), ("M", ctypes.c_int), ("N", ctypes.c_int)]
    gen = torch.Generator().manual_seed(M)
    shapes = [(8192, True, 8192), (1024, True, 1024), (96, False, 96), (64, True, 80), (256, False, 256)]
    jobs = (Job * len(shapes))()
    keep, want, outs = [], [], []
    for a, (N, masked, ld) in zip(jobs, shapes):
        dy = torch.randn(M, ld, generator=gen, dtype=torch.float64).float()
        mk = torch.randn(M, ld, generator=gen, dtype=torch.float64).float() if masked else None
        ref = dy.double()[:, :N]
        if masked:
            ref = torch.where(mk.double()[:, :N] > 0, ref, torch.zeros_like(ref))
        want.append(ref.sum(0))
        ddy, dmk = dev(dy), (dev(mk) if masked else None)
        db = torch.full((N,), 3.0, device="cuda")
        keep += [ddy, dmk, db]
        outs.append(db)
        a.dy, a.mask, a.db = ddy.data_ptr(), (dmk.data_ptr() if masked else None), db.data_ptr()
        a.ld, a.M, a.N = ld, M, N
    need = L.lib().ava_b200_bias_grads_ws_bytes(jobs, len(shapes))
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    L.call("ava_b200_bias_grads", jobs, len(shapes), ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    first = [o.clone() for o in outs]
    for j, (o, w) in enumerate(zip(outs, want)):
        got, ref = o.cpu().numpy().astype(np.float64), w.numpy()
        bad = np.flatnonzero(~(np.abs(got - ref) <= 1e-5 * np.abs(ref).max()))
        # says which job and how: columns never written (still 3.0), NaN, or wrong sums
        assert rel_err(got, ref) <= 1e-5, (
            "job %d %s: %d bad columns, %d still 3.0, %d NaN; first %s got %s want %s"
            % (j, shapes[j], bad.size, int((got[bad] == 3.0).sum()), int(np.isnan(got[bad]).sum()),
               bad[:8].tolist(), got[bad[:8]].tolist(), ref[bad[:8]].tolist()))
    L.call("ava_b200_bias_grads", jobs, len(shapes), ws.data_ptr(), need, stream())
    torch.cuda.synchronize()
    for o, f in zip(outs, first):
        assert torch.equal(o, f)


def test_adam_matches_torch(L):
    from oracle import vae_oracle
    n = 100003
    gen = torch.Generator().manual_seed(5)
    p = torch.randn(n, generator=gen)
    m = torch.zeros(n)
    v = torch.zeros(n)
    pad = (n + 3) // 4 * 4
    dp, dm, dv = [torch.zeros(pad, device="cuda") for _ in range(3)]
    dp[:n] = p.cuda()
    step = torch.zeros(1, device="cuda")
    p64, m64, v64 = p.double(), m.double(), v.double()
    for t in range(1, 4):
        g = torch.randn(n, generator=gen) * (10.0 ** (t - 2))
        dg = torch.zeros(pad, device="cuda")
        dg[:n] = g.cuda()
        L.call("ava_b200_adam_step", dp.data_ptr(), dg.data_ptr(), dm.data_ptr(), dv.data_ptr(), n,
               step.data_ptr(), 1e-3, 0.9, 0.999, 1e-8, 1.0, stream())
        vae_oracle.adam_step(p64, g.double(), m64, v64, t)
    torch.cuda.synchronize()
    assert step.item() == 3.0
    assert rel_err(dp[:n].cpu().numpy(), p64.numpy()) <= 1e-6
    assert rel_err(dm[:n].cpu().numpy(), m64.numpy()) <= 1e-6
    assert rel_err(dv[:n].cpu().numpy(), v64.numpy()) <= 1e-6


def test_bn_bookkeeping(L):
    from oracle import vae_oracle
    gen = torch.Generator().manual_seed(11)
    chans = [vae_oracle.bn_channels()[i + 1] for i in range(14)]
    counts = [1000 + 37 * i for i in range(14)]
    counts[3] = 0   # skipped layer
    stats = torch.zeros(14 * 64, dtype=torch.float64)
    dstats = torch.zeros(14 * 64, dtype=torch.float64)
    run = torch.zeros(14 * 64)
    means, variances = [], []
    for l, c in enumerate(chans):
        n = max(counts[l], 1)
        mean = torch.randn(c, generator=gen, dtype=torch.float64)
        var = torch.rand(c, generator=gen, dtype=torch.float64) + 0.1
        stats[l * 64:l * 64 + c] = mean * n
        stats[l * 64 + 32:l * 64 + 32 + c] = (var + mean * mean) * n
        dstats[l * 64:l * 64 + c] = torch.randn(c, generator=gen, dtype=torch.float64)
        dstats[l * 64 + 32:l * 64 + 32 + c] = torch.randn(c, generator=gen, dtype=torch.float64)
        run[l * 64:l * 64 + c] = torch.randn(c, generator=gen)
        run[l * 64 + 32:l * 64 + 32 + c] = torch.rand(c, generator=gen) + 0.5
        means.append(mean)
        variances.append(var)
    run0 = run.clone()
    dstat, ddstat, drun = stats.cuda(), dstats.cuda(), run.cuda()
    nbt = torch.full((14,), 4, dtype=torch.int64, device="cuda")
    hc = (ctypes.c_int * 14)(*chans)
    hn = (ctypes.c_longlong * 14)(*counts)
    rm_off = (ctypes.c_int * 14)(*[i * 64 for i in range(14)])
    rv_off = (ctypes.c_int * 14)(*[i * 64 + 32 for i in range(14)])
    L.call("ava_b200_bn_update_running", dstat.data_ptr(), hc, hn, drun.data_ptr(), rm_off, rv_off,
           nbt.data_ptr(), 0.1, stream())
    grads = torch.zeros(14 * 64, device="cuda")
    L.call("ava_b200_bn_param_grads", dstat.data_ptr(), ddstat.data_ptr(), hc, hn, grads.data_ptr(),
           rm_off, rv_off, stream())
    torch.cuda.synchronize()
    got, gg = drun.cpu(), grads.cpu()
    for l, c in enumerate(chans):
        sl_m, sl_v = slice(l * 64, l * 64 + c), slice(l * 64 + 32, l * 64 + 32 + c)
        if counts[l] == 0:
            assert torch.equal(got[sl_m], run0[sl_m]) and int(nbt[l]) == 4
            continue
        n = counts[l]
        assert int(nbt[l]) == 5
        want_m = 0.9 * run0[sl_m].double() + 0.1 * means[l]
        want_v = 0.9 * run0[sl_v].double() + 0.1 * variances[l] * n / (n - 1)
        assert rel_err(got[sl_m].numpy(), want_m.numpy()) <= 1e-6
        assert rel_err(got[sl_v].numpy(), want_v.numpy()) <= 1e-6
        invstd = 1.0 / torch.sqrt(variances[l] + 1e-5)
        assert rel_err(gg[sl_m].numpy(), (invstd * dstats[sl_v]).numpy()) <= 1e-6
        assert rel_err(gg[sl_v].numpy(), dstats[sl_m].numpy()) <= 1e-6


@pytest.mark.parametrize("precision,tol", [(2, 2e-5), (1, 3e-3)])
@pytest.mark.parametrize("M,N,K", [(128, 1024, 8192), (256, 8192, 1024), (128, 128, 32),
                                   (64, 1024, 8192), (64, 8192, 1024), (100, 256, 1024), (7, 1024, 256),
                                   (130, 8192, 1024), (1, 1024, 8192)])
def test_linear_tensor_core(L, precision, tol, M, N, K):
    """fc1/fc8-shaped layers on the tensor cores: the tcgen05 path when the batch tiles by 128,
    else the 64x64 tiled kernel with an mma.sync inner product (batch 64, ragged batches).
    precision 2 = 3xTF32 (fp32-level parity, tolerance 2e-5), precision 1 = single TF32
    (stated tolerance 3e-3)."""
    gen = torch.Generator().manual_seed(M + N + K + precision)
    x = (torch.randn(M, K, generator=gen, dtype=torch.float64) * 0.5).float().double()
    w = (torch.randn(N, K, generator=gen, dtype=torch.float64) / np.sqrt(K)).float().double()
    b = (torch.randn(N, generator=gen, dtype=torch.float64) * 0.1).float().double()
    x.requires_grad_(True)
    w.requires_grad_(True)
    b.requires_grad_(True)
    y_ref = F.relu(F.linear(x, w, b))
    dY = torch.randn(M, N, generator=gen, dtype=torch.float64).float().double()
    (y_ref * dY).sum().backward()
    dx_, dw_, db_, ddy = dev(x.detach()), dev(w.detach()), dev(b.detach()), dev(dY)
    y = torch.empty(M, N, device="cuda")
    ws_bytes = L.lib().ava_b200_linear_ws_bytes(M, N, K)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
    L.call("ava_b200_linear_fwd", dx_.data_ptr(), K, dw_.data_ptr(), db_.data_ptr(), y.data_ptr(), N,
           M, N, K, 1, 1, 0, 0, 0, 0, precision, ws.data_ptr(), ws_bytes, stream())
    gw = torch.full((N, K), 3.0, device="cuda")
    gb = torch.full((N,), 3.0, device="cuda")
    gx = torch.full((M, K), 3.0, device="cuda")
    # mask from the float64 reference so that a TF32 rounding flip cannot move the ReLU mask
    ymask = dev(y_ref.detach())
    L.call("ava_b200_linear_bwd_weight", ddy.data_ptr(), N, ymask.data_ptr(), dx_.data_ptr(), K,
           gw.data_ptr(), gb.data_ptr(), M, N, K, 1, 0, 0, 0, 0, precision, ws.data_ptr(), ws_bytes,
           stream())
    L.call("ava_b200_linear_bwd_data", ddy.data_ptr(), N, ymask.data_ptr(), dw_.data_ptr(),
           gx.data_ptr(), K, M, N, K, 1, 0, 0, 0, 0, precision, ws.data_ptr(), ws_bytes, stream())
    torch.cuda.synchronize()
    assert rel_err(y.cpu().numpy(), y_ref.detach().numpy()) <= tol
    assert rel_err(gw.cpu().numpy(), w.grad.numpy()) <= tol
    assert rel_err(gb.cpu().numpy(), b.grad.numpy()) <= 1e-5
    assert rel_err(gx.cpu().numpy(), x.grad.numpy()) <= tol
