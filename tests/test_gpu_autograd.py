"""Differentiable encode / decode / forward: the eval-mode BatchNorm backward kernels through the C ABI,
and the autograd functions of VAE.encode, VAE.decode and VAE.forward against the float64 oracle on the
GPU's ReLU pattern, in train and eval mode, plus the ownership rules of their activation sets."""
import ctypes
import importlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import vae_oracle
from tests.helpers import gpu_relu_masks, rel_err
from tests.test_gpu_kernels import LAYERS, dev, make_layer_inputs, stream

pytestmark = pytest.mark.gpu
PKG = "autoencoded-vocal-analysis_b200"
TOL = 1e-4
ctypes_int, ctypes_ll = ctypes.c_int, ctypes.c_longlong
ENC_MASKS = ["conv%d" % i for i in range(1, 8)] + ["fc1", "fc2", "fc3"]
DEC_MASKS = ["fc5", "fc6", "fc7", "fc8"] + ["convt%d" % i for i in range(1, 7)]


@pytest.fixture(scope="module")
def L():
    lib = importlib.import_module(PKG + "._lib")
    lib.lib()
    return lib


@pytest.fixture(scope="module")
def vae_mod():
    return importlib.import_module(PKG + ".models.vae")


def _guarded(shape, G=64):
    """A NaN-filled buffer with `shape` in its middle and G elements of guard band on either side."""
    n = int(np.prod(shape))
    buf = torch.full((n + 2 * G,), float("nan"), device="cuda")
    return buf, buf[G:G + n].view(shape)


def _guards_intact(buf, n, G=64):
    return bool(torch.isnan(buf[:G]).all()) and bool(torch.isnan(buf[G + n:]).all())


# ------------------------------------------------------------------------ kernels, eval mode
@pytest.mark.parametrize("mode", [0, 2, 6], ids=["fp32", "tf32x3", "tf32x3e"])
@pytest.mark.parametrize("l", range(14))
def test_bnconv_bwd_eval(L, l, mode):
    """Eval-mode BatchNorm backward of one fused layer (the _ex entries with train = 0) against float64
    autograd of F.batch_norm(training=False) -> conv / conv-transpose, with running statistics near the
    batch's own and far from them; outputs inside NaN guard bands."""
    name, ci, co, s, h, tr = LAYERS[l]
    L.call("ava_b200_set_conv_precision", mode)
    try:
        for B in (3, 64, 130):
            x, w, b, gamma, beta, _, _ = make_layer_inputs(l, B, 400 + l)
            near_m = x.mean(dim=(0, 2, 3)).float().double()
            near_v = x.var(dim=(0, 2, 3)).float().double()
            for rm, rv in ((near_m, near_v), ((near_m + 1.5).float().double(), (4.0 * near_v).float().double())):
                xr = x.clone().requires_grad_(True)
                wr, br = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
                gr, ber = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
                xn = F.batch_norm(xr, rm.clone(), rv.clone(), gr, ber, training=False, eps=1e-5)
                xn.retain_grad()
                if tr:
                    z = F.conv_transpose2d(xn, wr, br, stride=s, padding=1, output_padding=s - 1)
                else:
                    z = F.conv2d(xn, wr, br, stride=s, padding=1)
                ho = z.shape[-1]
                gen = torch.Generator().manual_seed(500 + l + B)
                dz = (torch.randn(z.shape, generator=gen, dtype=torch.float64) + 0.1).float().double()
                z.backward(dz)
                ddz, dx, dw_, dg, dbeta = dev(dz), dev(x), dev(w), dev(gamma), dev(beta)
                run = torch.zeros(64, device="cuda")
                run[:ci] = rm.float().cuda()
                run[32:32 + ci] = rv.float().cuda()
                tsums = torch.zeros(288, dtype=torch.float64, device="cuda")
                L.call("ava_b200_dz_border_sums", ddz.data_ptr(), B, co, ho, ho, 1 if (tr and s == 2) else 0,
                       tsums.data_ptr(), stream())
                ws = torch.empty(L.lib().ava_b200_bnconv_bwd_weight_ws(l, B), dtype=torch.uint8, device="cuda")
                gwb, gw = _guarded(tuple(w.shape))
                gbb, gb = _guarded((co,))
                dst = torch.zeros(64, dtype=torch.float64, device="cuda")
                L.call("ava_b200_bnconv_bwd_weight_ex", l, B, ddz.data_ptr(), dx.data_ptr(), dw_.data_ptr(),
                       dg.data_ptr(), dbeta.data_ptr(), None, run.data_ptr(), run.data_ptr() + 4 * 32, 0,
                       tsums.data_ptr(), gw.data_ptr(), gb.data_ptr(), dst.data_ptr(), ws.data_ptr(), stream())
                outs = {}
                for mask in (1, 0):
                    gib, gi = _guarded((B, ci, h, h))
                    L.call("ava_b200_bnconv_bwd_data_ex", l, B, ddz.data_ptr(), dw_.data_ptr(), dx.data_ptr(),
                           dg.data_ptr(), None, run.data_ptr() + 4 * 32, 0, None, mask, gi.data_ptr(), None,
                           stream())
                    outs[mask] = (gib, gi)
                # BatchNorm affine gradients of this layer (slot 0 of a 14-layer table; others skipped)
                grads_b, grads = _guarded((64,))
                chans = (ctypes_int * 14)(*([ci] + [1] * 13))
                counts = (ctypes_ll * 14)(*([B * h * h] + [0] * 13))
                offg = (ctypes_int * 14)(*([0] * 14))
                offb = (ctypes_int * 14)(*([32] * 14))
                offrv = (ctypes_int * 14)(*([32] * 14))
                L.call("ava_b200_bn_param_grads_ex", None, dst.data_ptr(), chans, counts, grads.data_ptr(), offg,
                       offb, run.data_ptr(), offrv, 0, stream())
                torch.cuda.synchronize()
                tag = (B, float(rm[0]))
                assert rel_err(gw.cpu().numpy(), wr.grad.numpy()) <= TOL, ("dw",) + tag
                assert rel_err(gb.cpu().numpy(), br.grad.numpy()) <= 1e-6, ("db",) + tag
                assert rel_err(outs[0][1].cpu().numpy(), xr.grad.numpy()) <= TOL, ("dx",) + tag
                assert rel_err(outs[1][1].cpu().numpy(), (xr.grad * (x > 0)).numpy()) <= TOL, ("dx masked",) + tag
                g_all = grads.cpu().numpy()
                # (cancellation-aware scale, as for the train-mode reductions in test_gpu_kernels.py)
                scale = max(float(xn.grad.abs().sum()) / ci, 1e-30)
                xc = (x - rm.view(1, -1, 1, 1)) / torch.sqrt(rv.view(1, -1, 1, 1) + 1e-5)
                gscale = max(float((xn.grad * xc).abs().sum()) / ci, 1e-30)
                assert np.abs(g_all[:ci] - gr.grad.numpy()).max() <= 1e-5 * gscale, ("dgamma",) + tag
                assert np.abs(g_all[32:32 + ci] - ber.grad.numpy()).max() <= 1e-5 * scale, ("dbeta",) + tag
                assert np.isnan(g_all[ci:32]).all() and np.isnan(g_all[32 + ci:]).all(), "unused channels written"
                for buf, t in ((gwb, gw), (gbb, gb), (grads_b, grads)) + tuple(outs.values()):
                    assert _guards_intact(buf, t.numel()), ("guard band",) + tag
    finally:
        L.call("ava_b200_set_conv_precision", 0)


@pytest.mark.parametrize("l", range(14))
def test_ex_train_is_the_old_entry(L, l):
    """The _ex entries with train = 1 are the existing entries, bit for bit."""
    name, ci, co, s, h, tr = LAYERS[l]
    B = 64
    L.call("ava_b200_set_conv_precision", 6)
    try:
        x, w, b, gamma, beta, rm, rv = make_layer_inputs(l, B, 600 + l)
        ho = h * 2 if (tr and s == 2) else (h // 2 if s == 2 else h)
        gen = torch.Generator().manual_seed(700 + l)
        dz = torch.randn(B, co, ho, ho, generator=gen).cuda()
        dx, dw_, dg, dbeta, drm, drv = dev(x), dev(w), dev(gamma), dev(beta), dev(rm), dev(rv)
        stats = torch.zeros(64, dtype=torch.float64, device="cuda")
        L.call("ava_b200_channel_stats", dx.data_ptr(), B, ci, h * h, stats.data_ptr(), stream())
        tsums = torch.zeros(288, dtype=torch.float64, device="cuda")
        L.call("ava_b200_dz_border_sums", dz.data_ptr(), B, co, ho, ho, 1 if (tr and s == 2) else 0,
               tsums.data_ptr(), stream())
        ws = torch.empty(L.lib().ava_b200_bnconv_bwd_weight_ws(l, B), dtype=torch.uint8, device="cuda")
        res = []
        for ex in (False, True):
            gw, gb = torch.empty_like(dw_), torch.empty(co, device="cuda")
            dst = torch.zeros(64, dtype=torch.float64, device="cuda")
            gi = torch.empty(B, ci, h, h, device="cuda")
            grads = torch.zeros(64, device="cuda")
            chans = (ctypes_int * 14)(*([ci] + [1] * 13))
            counts = (ctypes_ll * 14)(*([B * h * h] + [0] * 13))
            offg, offb = (ctypes_int * 14)(*([0] * 14)), (ctypes_int * 14)(*([32] * 14))
            if ex:
                L.call("ava_b200_bnconv_bwd_weight_ex", l, B, dz.data_ptr(), dx.data_ptr(), dw_.data_ptr(),
                       dg.data_ptr(), dbeta.data_ptr(), stats.data_ptr(), drm.data_ptr(), drv.data_ptr(), 1,
                       tsums.data_ptr(), gw.data_ptr(), gb.data_ptr(), dst.data_ptr(), ws.data_ptr(), stream())
                L.call("ava_b200_bnconv_bwd_data_ex", l, B, dz.data_ptr(), dw_.data_ptr(), dx.data_ptr(),
                       dg.data_ptr(), stats.data_ptr(), drv.data_ptr(), 1, dst.data_ptr(), 1, gi.data_ptr(), None,
                       stream())
                L.call("ava_b200_bn_param_grads_ex", stats.data_ptr(), dst.data_ptr(), chans, counts,
                       grads.data_ptr(), offg, offb, drv.data_ptr(), offg, 1, stream())
            else:
                L.call("ava_b200_bnconv_bwd_weight", l, B, dz.data_ptr(), dx.data_ptr(), dw_.data_ptr(),
                       dg.data_ptr(), dbeta.data_ptr(), stats.data_ptr(), tsums.data_ptr(), gw.data_ptr(),
                       gb.data_ptr(), dst.data_ptr(), ws.data_ptr(), stream())
                L.call("ava_b200_bnconv_bwd_data", l, B, dz.data_ptr(), dw_.data_ptr(), dx.data_ptr(),
                       dg.data_ptr(), stats.data_ptr(), dst.data_ptr(), 1, gi.data_ptr(), None, stream())
                L.call("ava_b200_bn_param_grads", stats.data_ptr(), dst.data_ptr(), chans, counts,
                       grads.data_ptr(), offg, offb, stream())
            torch.cuda.synchronize()
            res.append((gw, gb, gi, grads))
        # (dstats are fp64 atomics: the two runs may add in another order, so dx and dgamma, which read
        # them, are compared to the last bits; dw and db come from the deterministic two-stage sums)
        assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
        assert rel_err(res[1][2].cpu().numpy(), res[0][2].cpu().numpy()) <= 1e-6
        assert rel_err(res[1][3].cpu().numpy(), res[0][3].cpu().numpy()) <= 1e-6
    finally:
        L.call("ava_b200_set_conv_precision", 0)


def test_seam_kernels(L):
    B, Z = 37, 32
    g = torch.Generator().manual_seed(5)
    dmu, du, dd, d = (torch.randn(B, Z, generator=g).cuda() for _ in range(4))
    out = torch.full((B, 3 * Z), float("nan"), device="cuda")
    L.call("ava_b200_latent_heads_grad", dmu.data_ptr(), du.data_ptr(), dd.data_ptr(), d.data_ptr(), B, Z,
           out.data_ptr(), stream())
    torch.cuda.synchronize()
    assert torch.equal(out, torch.cat([dmu, du, dd * d], dim=1))
    L.call("ava_b200_latent_heads_grad", None, du.data_ptr(), None, None, B, Z, out.data_ptr(), stream())
    torch.cuda.synchronize()
    assert torch.equal(out, torch.cat([torch.zeros_like(dmu), du, torch.zeros_like(dd)], dim=1))
    x, xr, de = (torch.randn(B, 128, 128, generator=g).cuda() for _ in range(3))
    dx = torch.empty_like(x)
    L.call("ava_b200_recon_input_grad", de.data_ptr(), x.data_ptr(), xr.data_ptr(), B * 128 * 128, 10.0,
           dx.data_ptr(), stream())
    torch.cuda.synchronize()
    ref = de.double() - 10.0 * (xr.double() - x.double())
    assert rel_err(dx.cpu().numpy(), ref.cpu().numpy()) <= 1e-6


# ---------------------------------------------------------------------------- model level
def _build(vae_mod, seed, precision="auto", **kw):
    model = vae_mod.VAE(save_dir='', device_name='cuda', precision=precision, **kw)
    model.load_flat_state(vae_oracle.make_params(seed))
    return model


def _oracle(objective, P, inputs, dtype):
    """Gradients of objective(Q, inputs) w.r.t. the 80 parameters and the inputs, on the GPU in `dtype`
    (float32 without TF32: the reference arithmetic's own rounding)."""
    keys = [k for k, _ in vae_oracle.param_order()]
    Q = {k: v.to(device="cuda", dtype=dtype if v.is_floating_point() else v.dtype) for k, v in P.items()}
    for k in keys:
        Q[k] = Q[k].clone().requires_grad_(True)
    ins = [t.to(device="cuda", dtype=dtype).clone().requires_grad_(True) for t in inputs]
    prev = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    try:
        obj = objective(Q, ins)
        gs = torch.autograd.grad(obj, [Q[k] for k in keys] + ins, allow_unused=True)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = prev
    out = dict(zip(keys, gs[:len(keys)]))
    return out, list(gs[len(keys):])


def _check(got_params, got_inputs, objective, P, inputs, tag):
    """Every gradient within max(1e-4, 3 x the float32 oracle's error) of the float64 oracle (max-norm)."""
    g64, i64 = _oracle(objective, P, inputs, torch.float64)
    g32, i32 = _oracle(objective, P, inputs, torch.float32)
    worst = 0.0
    for k, ref in list(g64.items()) + [("input%d" % i, t) for i, t in enumerate(i64)]:
        got = got_params.get(k) if not k.startswith("input") else got_inputs[int(k[5:])]
        if ref is None:
            assert got is None, (tag, k, "gradient where none is due")
            continue
        assert got is not None, (tag, k, "missing gradient")
        r32 = g32[k] if not k.startswith("input") else i32[int(k[5:])]
        ref_n = ref.detach().cpu().numpy()
        bar = max(TOL, 3.0 * rel_err(r32.detach().double().cpu().numpy(), ref_n))
        err = rel_err(got.detach().double().cpu().numpy().reshape(ref_n.shape), ref_n)
        worst = max(worst, err / bar)
        assert err <= bar, (tag, k, err, bar)
    print("%s: worst error / bar %.2f" % (tag, worst))


def _flips(masks, P, x, train, names):
    """ReLU units on the other side of zero than the float64 oracle's own forward, and the float32
    oracle's count on the same inputs."""
    counts = []
    for dt in (torch.float64, torch.float32):
        acts = {}
        Q = {k: v.to(device="cuda", dtype=dt if v.is_floating_point() else v.dtype) for k, v in P.items()}
        with torch.no_grad():
            mu, u, d = vae_oracle.encode(Q, x.to("cuda", dt), train, None, acts)
            vae_oracle.decode(Q, mu, train, None, acts)
        counts.append(acts)
    a64, a32 = counts
    f32 = sum(int(((a32[n] > 0) != (a64[n] > 0)).sum()) for n in names)
    f = sum(int((masks[n].cuda() != (a64[n].reshape(masks[n].shape) > 0)).sum()) for n in names)
    return f, f32


CASES = [(B, train, prec) for B in (7, 64, 130) for train in (True, False) for prec in ("auto", "fp32")] + \
    [(1024, True, "auto"), (1024, False, "auto")]


@pytest.mark.parametrize("B,train,precision", CASES)
@pytest.mark.parametrize("kind", ["encode", "decode", "forward", "compose"])
def test_model_autograd(vae_mod, kind, B, train, precision):
    seed = 3
    model = _build(vae_mod, seed, precision)
    model.train(train)
    P = vae_oracle.make_params(seed)
    x = vae_oracle.make_input(seed, B).cuda().requires_grad_(True)
    ew, ed = (t.cuda() for t in vae_oracle.make_noise(seed, B))
    gen = torch.Generator().manual_seed(B)
    names = dict(model.named_parameters())
    tag = "%s B=%d %s %s" % (kind, B, "train" if train else "eval", precision)
    if kind == "encode":
        seeds = [torch.randn(B, 32, generator=gen).cuda() for _ in range(3)]
        mu, u, d = model.encode(x)
        masks = gpu_relu_masks(model._cur)
        ((mu * seeds[0]).sum() + (u.squeeze(-1) * seeds[1]).sum() + (d * seeds[2]).sum()).backward()

        def objective(Q, ins):
            m, uu, dd = vae_oracle.encode(Q, ins[0], train, None, None, masks_dev)
            return (m * seeds[0]).sum() + (uu.squeeze(-1) * seeds[1]).sum() + (dd * seeds[2]).sum()
        inputs, mask_names = [x.detach()], ENC_MASKS
        got_in = [x.grad]
    elif kind == "decode":
        z = torch.randn(B, 32, generator=gen).cuda().requires_grad_(True)
        seed_x = torch.randn(B, 128 * 128, generator=gen).cuda()
        xr = model.decode(z)
        masks = gpu_relu_masks(model._cur)
        (xr * seed_x).sum().backward()

        def objective(Q, ins):
            return (vae_oracle.decode(Q, ins[0], train, None, None, masks_dev) * seed_x).sum()
        inputs, mask_names = [z.detach()], DEC_MASKS
        got_in = [z.grad]
    elif kind == "forward":
        loss = model(x, noise=(ew, ed))
        masks = gpu_relu_masks(model._cur)
        (2.5 * loss).backward()

        def objective(Q, ins):
            return 2.5 * vae_oracle.forward(Q, ins[0], ew, ed, 10.0, train, None, None, masks_dev)["loss"]
        inputs, mask_names = [x.detach()], ENC_MASKS + DEC_MASKS
        got_in = [x.grad]
    else:
        mu, u, d = model.encode(x)
        m_enc = gpu_relu_masks(model._cur)
        zz = mu + u.squeeze(-1) * ew + torch.sqrt(d) * ed
        xr = model.decode(zz)
        m_dec = gpu_relu_masks(model._cur)
        masks = {**{k: m_enc[k] for k in ENC_MASKS}, **{k: m_dec[k] for k in DEC_MASKS}}
        (0.5 * ((xr - x.reshape(B, -1)) ** 2).sum() + (mu * mu).sum()).backward()

        def objective(Q, ins):
            m, uu, dd = vae_oracle.encode(Q, ins[0], train, None, None, masks_dev)
            r = vae_oracle.decode(Q, m + uu.squeeze(-1) * ew + torch.sqrt(dd) * ed, train, None, None, masks_dev)
            return 0.5 * ((r - ins[0].reshape(B, -1)) ** 2).sum() + (m * m).sum()
        inputs, mask_names = [x.detach()], ENC_MASKS + DEC_MASKS
        got_in = [x.grad]
    torch.cuda.synchronize()
    masks_dev = {k: masks[k].cuda() for k in mask_names}
    got = {k: p.grad for k, p in names.items()}
    _check(got, got_in, objective, P, inputs, tag)
    if kind in ("encode", "forward", "compose"):
        f, f32 = _flips(masks, P, x.detach(), train, [n for n in mask_names if n in ENC_MASKS])
        assert f <= max(16, 4 * f32), (tag, f, f32)


# ------------------------------------------------------------------------------- semantics
def test_input_grad_leaves_param_grads(vae_mod):
    x = vae_oracle.make_input(1, 64).cuda()
    noise = tuple(t.cuda() for t in vae_oracle.make_noise(1, 64))
    res = []
    for want_x in (False, True):
        model = _build(vae_mod, 1)
        model.train()
        xx = x.clone().requires_grad_(want_x)
        model(xx, noise=noise).backward()
        res.append({k: p.grad.clone() for k, p in model.named_parameters()})
        assert (xx.grad is not None) == want_x
    for k in res[0]:
        assert rel_err(res[1][k].cpu().numpy(), res[0][k].cpu().numpy()) <= 1e-6, k


def test_eval_backward_keeps_running_buffers(vae_mod):
    model = _build(vae_mod, 2)
    model.eval()
    run, nbt = model._flat_run.clone(), model._nbt.clone()
    x = vae_oracle.make_input(2, 16).cuda().requires_grad_(True)
    model(x).backward()
    mu, u, d = model.encode(x)
    (mu.sum() + d.sum()).backward()
    model.decode(mu.detach().requires_grad_(True)).sum().backward()
    torch.cuda.synchronize()
    assert torch.equal(model._flat_run, run) and torch.equal(model._nbt, nbt)


def test_eval_backward_uses_the_forwards_running_buffers(vae_mod):
    """Eval forward, then a train-mode forward that moves the running buffers, then the first graph's
    backward: the gradient is the one of the statistics the forward normalised with."""
    seed, B = 4, 16
    model = _build(vae_mod, seed)
    P = vae_oracle.make_params(seed)
    x = vae_oracle.make_input(seed, B).cuda().requires_grad_(True)
    ew, ed = (t.cuda() for t in vae_oracle.make_noise(seed, B))
    model.eval()
    loss = model(x, noise=(ew, ed))
    masks = {k: v.cuda() for k, v in gpu_relu_masks(model._cur).items()}
    model.train()
    with torch.no_grad():
        model(vae_oracle.make_input(seed + 1, B).cuda() * 3.0)
    assert not torch.equal(model.bn3.running_mean.cpu(), P["bn3.running_mean"])
    loss.backward()
    torch.cuda.synchronize()

    def objective(Q, ins):
        return vae_oracle.forward(Q, ins[0], ew, ed, 10.0, False, None, None, masks)["loss"]
    _check({k: p.grad for k, p in model.named_parameters()}, [x.grad], objective, P, [x.detach()], "snapshot")


def test_frozen_model_fills_only_input_grad(vae_mod):
    model = _build(vae_mod, 5)
    model.eval()
    model.requires_grad_(False)
    x = vae_oracle.make_input(5, 8).cuda().requires_grad_(True)
    model(x).backward()
    assert x.grad is not None and torch.isfinite(x.grad).all()
    assert all(p.grad is None for p in model.parameters())
    mu, _, _ = model.encode(x)
    assert mu.requires_grad
    with torch.no_grad():
        assert not model.encode(x)[0].requires_grad


def test_double_backward_raises(vae_mod):
    model = _build(vae_mod, 6)
    model.train()
    x = vae_oracle.make_input(6, 8).cuda().requires_grad_(True)
    loss = model(x)
    gx, = torch.autograd.grad(loss, x, create_graph=True)
    with pytest.raises(RuntimeError):
        gx.sum().backward()
    loss = model(x)
    loss.backward(retain_graph=True)
    with pytest.raises(RuntimeError, match="already run"):
        loss.backward()


# ------------------------------------------------------------------------------- ownership
def test_two_forwards_one_backward(vae_mod):
    seed, B = 7, 32
    model = _build(vae_mod, seed)
    model.train()
    P = vae_oracle.make_params(seed)
    xs = [vae_oracle.make_input(seed + i, B).cuda().requires_grad_(True) for i in range(2)]
    noise = [tuple(t.cuda() for t in vae_oracle.make_noise(seed + i, B)) for i in range(2)]
    losses, masks = [], []
    for x, nz in zip(xs, noise):
        losses.append(model(x, noise=nz))
        masks.append({k: v.cuda() for k, v in gpu_relu_masks(model._cur).items()})
    (losses[0] + losses[1]).backward()
    torch.cuda.synchronize()

    def objective(Q, ins):
        return sum(vae_oracle.forward(Q, ins[i], noise[i][0], noise[i][1], 10.0, True, None, None, masks[i])["loss"]
                   for i in range(2))
    _check({k: p.grad for k, p in model.named_parameters()}, [x.grad for x in xs], objective, P,
           [x.detach() for x in xs], "two forwards")


def test_train_step_between_forward_and_backward(vae_mod):
    """A captured train_step graph at the same batch size runs between a forward and its backward: neither
    touches the other's activations (learning rate 0, so the weights the backward reads stay put)."""
    seed, B = 8, 64
    P = vae_oracle.make_params(seed)
    models = [_build(vae_mod, seed) for _ in range(2)]
    steps = [vae_oracle.make_input(seed + 10 + i, B).cuda() for i in range(4)]
    snoise = [tuple(t.cuda() for t in vae_oracle.make_noise(seed + 10 + i, B)) for i in range(4)]
    for m in models:
        m.train()
        m.optimizer.param_groups[0]["lr"] = 0.0
        for i in range(3):                       # the third step is captured as a CUDA graph
            m.train_step(steps[i], noise=snoise[i])
    x = vae_oracle.make_input(seed, B).cuda().requires_grad_(True)
    ew, ed = (t.cuda() for t in vae_oracle.make_noise(seed, B))
    m = models[0]
    loss = m(x, noise=(ew, ed))
    masks = {k: v.cuda() for k, v in gpu_relu_masks(m._cur).items()}
    l_step = [mm.train_step(steps[3], noise=snoise[3]).clone() for mm in models]
    g_step = [mm._flat_g.clone() for mm in models]
    torch.cuda.synchronize()
    assert abs(float(l_step[0]) - float(l_step[1])) <= 1e-6 * abs(float(l_step[1]))
    assert rel_err(g_step[0].cpu().numpy(), g_step[1].cpu().numpy()) <= 1e-6
    m.zero_grad()
    loss.backward()
    torch.cuda.synchronize()

    def objective(Q, ins):
        return vae_oracle.forward(Q, ins[0], ew, ed, 10.0, True, None, None, masks)["loss"]
    _check({k: p.grad for k, p in m.named_parameters()}, [x.grad], objective, P, [x.detach()], "train_step between")


def test_memory_steady_in_a_loop(vae_mod):
    model = _build(vae_mod, 9)
    model.train()
    x = vae_oracle.make_input(9, 64).cuda().requires_grad_(True)
    seen = {}
    for it in range(1, 11):
        loss = model(x)
        loss.backward()
        mu, u, d = model.encode(x)
        (mu.sum() + model.decode(mu).sum()).backward()
        torch.cuda.synchronize()
        seen[it] = torch.cuda.memory_allocated()
    assert seen[3] == seen[10], seen
